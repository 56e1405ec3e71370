#!/usr/bin/env python3
"""bench.py -- throughput of the stereo front-end hot path on synthetic data, one JSON line per run.

  python bench.py [--config c1|c2|c3|c4|c5] [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--dump-outputs writes the results of the last timed step as .npy files; the inputs are seeded, so two builds run with the
same arguments can be compared output for output.

Configurations (BASELINE.json `configs`, SURVEY.md section 8):
  c1  one KITTI-00-shaped 1241x376 pair per step, maxCorners 1000 (the reference's own CPU-runnable case)
  c2  (default, the configuration the metric is quoted on) 4096 pairs of 1241x376 per GPU and step, maxCorners 2000;
      every rank owns its own batch -- weak scaling, no collective on the data path
  c3  vi_sensor 752x480 SEQUENCE: projection-window tracking (trackManual stages 1-3) of the landmark set that the
      per-frame loop of CTrackerGT builds up (~3000 landmarks), state fed forward; ranks run independent replicas
  c4  kitti_11_12-shaped batch of 32768 pairs of 1226x370 cut into contiguous frame ranges over the ranks
      (strong scaling: the total is fixed), maxCorners 1000
  c5  stress: 3840x1080 pairs, maxCorners 10000, 1000 px scan-line range

Per line:
  value        whole-job frames/s with inputs and outputs resident in HBM (svi_stereo_frames_device), CUDA events on the
               launching stream, barrier + synchronize on both sides, max over ranks  (c3: the host-buffer call, see there)
  e2e          the same metric through the host-buffer C-ABI call (svi_stereo_frames / svi_track_landmarks): pinned host
               images -> device -> results back in pinned host memory, every step
  roofline     the dominant kernel's algorithmic bytes per launch / its exclusive launch duration (one extra profiled
               step with all chunks on one stream, CUDA events of the library) against the measured HBM peak, plus the
               per-kernel record and the unit that actually binds (shared-memory pipe, from the committed ncu capture)
  cpu_baseline the C restatement of the reference CPU path (oracle/svi_oracle.c) timed on this box's host cores on a
               bounded sample of the same frames -- and the parity gate: GPU results == CPU results on that sample
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import sys
import threading
import time
from types import SimpleNamespace

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True   # a run leaves the tree as build() left it (it may be read-only)

BYTES_PER_KEYPOINT = 113  # uvL 8 + uvR 8 + xyz 24 + descL 32 + descR 32 + dist 4 + idx 4 + status 1
CALIB = ROOT / "tests" / "golden" / "calib"
DTYPE = "f32+f64 (Harris/triangulation), u8/u16/u32 (BRIEF, Hamming)"

CONFIGS = {
    "c1": dict(calib="kitti_00", max_corners=1000, frames=1, steps=200, scaling="weak", seed=0,
               what="single KITTI-00-shaped synthetic 1241x376 pair per step, maxCorners 1000 (BASELINE.json configs[0])"),
    "c2": dict(calib="kitti_00", max_corners=2000, frames=4096, steps=5, scaling="weak", seed=1000,
               what="KITTI-00-shaped synthetic batch of 4096 stereo pairs per GPU at 1241x376, maxCorners 2000 (BASELINE.json configs[1])"),
    "c3": dict(calib="vi_sensor", max_corners=1000, frames=60, steps=3, scaling="weak", seed=4000,
               what="vi_sensor 752x480 synthetic sequence, trackManual stages 1-3 with landmark state fed forward (BASELINE.json configs[2])"),
    "c4": dict(calib="kitti_11_12", max_corners=1000, frames=32768, steps=3, scaling="strong", seed=2000,
               what="kitti_11_12-shaped synthetic batch of 32768 stereo pairs at 1226x370 partitioned by frame over the GPUs, "
                    "maxCorners 1000 (BASELINE.json configs[3])"),
    "c5": dict(calib="kitti_00", size=(3840, 1080), max_corners=10000, frames=16, steps=5, scaling="weak", seed=3000, search_range=1000.0,
               max_candidates=131072, d_max=900,
               what="stress: synthetic 3840x1080 pairs, maxCorners 10000, 1000 px scan-line range (BASELINE.json configs[4])"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=None, help="override the configuration's frames per step")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--device-only", action="store_true", help="tuning aid: only the device-resident measurement; not a bench line")
    ap.add_argument("--device-order", default=None, help="comma list: CUDA device of local rank i (placement experiments)")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not bind the rank to its GPU's NUMA node (placement experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 / float64, "
                         "under 64 MB: a fixed sample of the frames of a larger batch); rank 0 only")
    a = ap.parse_args()
    a.cfg = dict(CONFIGS[a.config])
    if a.frames is not None:
        a.cfg["frames"] = a.frames
    if a.steps is None:
        a.steps = a.cfg["steps"]
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


# ----------------------------------------------------------------------------- --dump-outputs
# svi_stereo_result field -> the name of the same array in run_batch's output tensors
RESULT_FIELDS = {"n_keypoints": "n_kp", "n_detected": "n_det", "uv_left": "uv_l", "uv_right": "uv_r", "xyz_left": "xyz",
                 "desc_left": "dl", "desc_right": "dr", "distance": "dist", "match_index": "idx", "status": "st"}
DUMP_BYTES = 60_000_000   # the arrays of the sampled frames; the .npy headers and per-frame counts stay well inside 64 MB


def dump_frame_sample(n_frames: int, cap: int):
    """Frames whose results --dump-outputs writes: all of them when they fit DUMP_BYTES, else a fixed seeded sample."""
    import numpy as np
    per_frame = cap * (2 * 4 + 2 * 4 + 3 * 8 + 2 * 32 * 4 + 3 * 4)   # uv x2, xyz, two descriptors (one float per byte), distance, index, status
    n = min(n_frames, max(1, DUMP_BYTES // per_frame))
    return np.arange(n_frames) if n == n_frames else np.sort(np.random.default_rng(0).choice(n_frames, n, replace=False))


def write_stereo_dump(out_dir, r: dict, frames) -> None:
    """svi_stereo_result arrays of the given frames (field names of include/svi_gpu.h) as float32, xyz as float64; every
    integer converts exactly.  What the C API leaves unspecified is written as 0: the slots past n_keypoints, and uv_right,
    xyz_left and desc_right of key-points whose status is not SVI_OK."""
    import numpy as np
    cap = r["status"].shape[1]
    live = np.arange(cap)[None, :] < r["n_keypoints"][:, None]
    matched = live & (r["status"] == 0)
    out = {"frame_index": np.asarray(frames, np.float64)}
    for k in ("n_keypoints", "n_detected"):
        out[k] = r[k].astype(np.float64)
    for k in ("uv_left", "uv_right", "xyz_left", "desc_left", "desc_right", "distance", "match_index", "status"):
        a = r[k].astype(np.float64 if k == "xyz_left" else np.float32)
        a[~(matched if k in ("uv_right", "xyz_left", "desc_right") else live)] = 0
        out[k] = a
    write_arrays(out_dir, out)


def write_sequence_dump(out_dir, trk) -> None:
    """The tracker after a whole sequence: its landmark state (one row per active landmark) and its per-frame record
    (tracked, visible, new, active, motion scaling, landmarks per tracking stage 0-5), all float64 (exact)."""
    import numpy as np
    out = {f"landmark_{k}": np.asarray(v, np.float64) for k, v in trk.s.items()}
    out["frame_log"] = np.array([[r["tracked"], r["visible"], r["new"], r["active"], r["scaling"], *r["stages"]] for r in trk.log], np.float64)
    write_arrays(out_dir, out)


def write_arrays(out_dir, arrays: dict) -> None:
    import numpy as np
    d = pathlib.Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", np.ascontiguousarray(a))


def cameras(cfg):
    from svi_mapper_b200 import load_camera
    cl, cr = load_camera(str(CALIB / f"{cfg['calib']}_left.txt")), load_camera(str(CALIB / f"{cfg['calib']}_right.txt"))
    if "size" in cfg:   # the stress frame keeps the KITTI-00 projection matrices on a larger image
        W, H = cfg["size"]
        cl, cr = SimpleNamespace(width=W, height=H, P=cl.P), SimpleNamespace(width=W, height=H, P=cr.P)
    return cl, cr


def frontend_kwargs(cfg):
    kw = dict(max_corners=cfg["max_corners"])
    if "search_range" in cfg:
        kw["search_range_px"] = cfg["search_range"]
    if "max_candidates" in cfg:
        kw["max_candidates"] = cfg["max_candidates"]
    return kw


def oracle_config(co, cams, cfg):
    return co.make_config(cams[0], cams[1], max_corners=cfg["max_corners"], search_range=cfg.get("search_range", 60.0))


def measured_hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_kernel_metrics():
    """Per-kernel counters of the committed ncu --set full capture (tools/ncu_summary.py): DRAM bytes per launch,
    shared-memory pipe / ALU / FMA / issue utilisation.  They describe the C2 launch shape (64 frames of 1241x376)."""
    p = ROOT / "profiles" / "r2_kernel_metrics.json"
    try:
        return json.loads(p.read_text())
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def stop(self) -> dict:
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def bind_to_gpu_numa_node(index: int) -> str:
    """Bind this process to the CPUs next to its GPU (NVML's ideal affinity) BEFORE any pinned buffer is allocated, so that
    the staging memory of every rank lives on the NUMA node its PCIe root port hangs off -- with all ranks on one node the
    host-to-device streams of a multi-GPU run meet on the inter-socket link."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        cpus = sorted(os.sched_getaffinity(0))
        return f"{len(cpus)} cpus [{cpus[0]}..{cpus[-1]}]"
    except Exception as e:   # no NVML / not permitted: run unbound
        return f"unbound ({type(e).__name__})"


def metric_name(name, cams):
    if name == "c3":
        return (f"tracked stereo frames/sec (projection-window landmark tracking, trackManual stages 1-3 + re-detection) "
                f"at {cams[0].width}x{cams[0].height}")
    return f"stereo frames/sec (detect+describe+match+triangulate) at {cams[0].width}x{cams[0].height}"


# ----------------------------------------------------------------------------- CPU arm (reference / baseline)
def load_oracle():
    """The checker built with -march=native for this host, as the reference builds itself, in a temporary directory so that
    the tree stays as build() left it; the portable build of build() when that fails.  Returns (module, `native` argument)."""
    import tempfile
    from oracle import c_oracle as co
    with tempfile.TemporaryDirectory(prefix="svi_oracle_") as d:
        try:
            native = co.build(native=True, out=pathlib.Path(d) / "libsvi_oracle_native.so")
            co.load(native)   # mapped (and cached by path) before the directory goes
        except Exception:
            native = False
    return co, native


def cpu_stereo_fps(co, native, ocfg, L, R, target_seconds, threads):
    """(fps all threads, fps one thread, n_sample, results) of the C restatement on the first frames of (L, R)."""
    t0 = time.perf_counter()
    co.stereo_frames(ocfg, L[:1], R[:1], n_threads=1, native=native)
    t_one = time.perf_counter() - t0
    n = int(max(min(threads, len(L)), min(len(L), target_seconds * threads / max(t_one, 1e-3))))
    n = max(1, min(n, len(L)))
    t0 = time.perf_counter()
    out = co.stereo_frames(ocfg, L[:n], R[:n], n_threads=threads, native=native)
    t_all = time.perf_counter() - t0
    return n / t_all, 1.0 / t_one, n, out


def stereo_parity(ref, got, n_frames):
    """GPU results (dict of (F, cap, ...) arrays) == CPU restatement on the first n_frames frames; xyz within 1e-5 relative."""
    import numpy as np
    ok = True
    for f in range(n_frames):
        k = int(ref["n_keypoints"][f])
        ok &= k == int(got["n_kp"][f])
        if not ok:
            break
        for a, b in (("uv_left", "uv_l"), ("desc_left", "dl"), ("status", "st"), ("distance", "dist"), ("match_index", "idx")):
            ok &= bool(np.array_equal(ref[a][f, :k], got[b][f, :k]))
        good = ref["status"][f, :k] == 0
        ok &= bool(np.array_equal(ref["uv_right"][f, :k][good], got["uv_r"][f, :k][good]))
        ok &= bool(np.array_equal(ref["desc_right"][f, :k][good], got["dr"][f, :k][good]))
        ok &= bool(np.allclose(ref["xyz_left"][f, :k][good], got["xyz"][f, :k][good], rtol=1e-5, atol=0))
    return bool(ok)


class CpuSequenceBackend:
    """SequenceTracker backend over the C restatement (trackManual + addNewLandmarks), with its own clock."""

    def __init__(self, co, native, ocfg, threads):
        from oracle import frontend_np as onp
        self.co, self.native, self.cfg, self.threads, self.onp, self.seconds = co, native, ocfg, threads, onp, 0.0

    def track(self, L, R, T, s, scaling, size):
        t0 = time.perf_counter()
        r = self.co.track_landmarks(self.cfg, L, R, T, s["xyz_w"], s["last_desc_l"], s["last_desc_r"], s["last_disp"], size, scaling,
                                    uv_reference_left=s["uv_ref"], desc_reference_left=s["ref_desc_l"],
                                    T_left_to_world_at_detection=s["T_det"], n_threads=self.threads, native=self.native)
        self.seconds += time.perf_counter() - t0
        return r

    def add_new(self, L, R, centres):
        t0 = time.perf_counter()
        m = self.onp.mask_active_landmarks(L.shape[1], L.shape[0], centres)[None] if len(centres) else None
        r = self.co.frame(self.co.stereo_frames(self.cfg, L, R, masks=m, n_threads=1, native=self.native), 0)
        self.seconds += time.perf_counter() - t0
        return r


def run_reference(args, rank: int):
    """--impl reference: the reference's own CPU algorithm (C restatement; the reference binary cannot be built here) on
    the host cores, every step a bounded sample of the configuration's workload."""
    if rank != 0:
        return
    import numpy as np
    from svi_mapper_b200.synth import stereo_pair
    cfg = args.cfg
    cams = cameras(cfg)
    co, native = load_oracle()
    threads = co.host_threads()
    ocfg = oracle_config(co, cams, cfg)
    W, H = cams[0].width, cams[0].height
    build = "-march=native" if native else "x86-64-v3"
    extra = {}
    if args.config == "c3":
        from svi_mapper_b200.sequence import SequenceTracker, render_sequence
        n = min(cfg["frames"], 24)
        L, R, T = render_sequence(cams[0], cams[1], n, cfg["seed"])
        steps = args.steps
        t_sum, lm_sum = 0.0, 0
        for _ in range(steps):
            be = CpuSequenceBackend(co, native, ocfg, threads)
            trk = SequenceTracker(be, cams[0])
            for t in range(n):
                lm_sum += trk.process(L[t], R[t], T[t])["tracked"]
            t_sum += be.seconds
        if args.dump_outputs:
            write_sequence_dump(args.dump_outputs, trk)
        fps = steps * n / t_sum
        sample = (f"first {n} frames of the sequence per step x {steps} steps, landmark-parallel over {threads} threads, "
                  f"{build} build of oracle/svi_oracle.c")
        extra = {"landmarks_per_s": lm_sum / t_sum}
        ms_step = t_sum / steps * 1e3
    else:
        big = W * H > 2_000_000
        n_unique = 2 if big else min(8, max(2, threads))
        pairs = [stereo_pair(W, H, cfg["seed"] + i, d_max=cfg.get("d_max", 55)) for i in range(n_unique)]
        sample_n = max(2, min(threads, 4)) if big else max(threads, 8)
        L = np.stack([pairs[i % n_unique][0] for i in range(sample_n)])
        R = np.stack([pairs[i % n_unique][1] for i in range(sample_n)])
        steps = args.steps
        for _ in range(min(args.warmup, 1)):
            co.stereo_frames(ocfg, L, R, n_threads=threads, native=native)
        t0 = time.perf_counter()
        for _ in range(steps):
            out = co.stereo_frames(ocfg, L, R, n_threads=threads, native=native)
        dt = time.perf_counter() - t0
        if args.dump_outputs:
            frames = dump_frame_sample(sample_n, cfg["max_corners"])
            write_stereo_dump(args.dump_outputs, {k: v[frames] for k, v in out.items()}, frames)
        fps = sample_n * steps / dt
        sample = f"{sample_n} frames/step x {steps} steps, {min(threads, sample_n)} threads (one frame per thread), {build} build of oracle/svi_oracle.c"
        ms_step = dt / steps * 1e3
    line = {"impl": "reference", "metric": metric_name(args.config, cams), "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": cfg["what"] + "; bounded sample per step on the host CPU", "name": args.config},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample, **extra},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm: batches (c1, c2, c4, c5)
def run_batch(args, rank, world, dev_index):
    import numpy as np
    import torch
    import torch.distributed as dist

    from svi_mapper_b200 import StereoFrontend, _lib, frame_range
    from svi_mapper_b200.synth import stereo_frames_range_torch

    cfg = args.cfg
    cams = cameras(cfg)
    W, H, cap = cams[0].width, cams[0].height, cfg["max_corners"]
    dev = torch.device("cuda", dev_index)
    if cfg["scaling"] == "strong":
        f_lo, f_hi = frame_range(cfg["frames"], world, rank)            # contiguous range of the fixed batch
    else:
        f_lo, f_hi = rank * cfg["frames"], (rank + 1) * cfg["frames"]    # every rank owns its own batch
    F = f_hi - f_lo
    fe = StereoFrontend(cams[0], cams[1], device=dev_index, **frontend_kwargs(cfg))
    fcfg = fe.config()
    kernels_per_chunk = fe.kernels_per_chunk(F)
    frame_bytes = 2 * W * H + BYTES_PER_KEYPOINT * cap   # SURVEY.md 8(d): every input byte once + 113 B per key-point slot

    # synthetic frames generated on the device; frame i has the same content whatever the partition
    dL, dR = stereo_frames_range_torch(f_lo, F, W, H, cfg["seed"], device=dev, d_max=cfg.get("d_max", 55))
    torch.cuda.synchronize()

    def outputs(n, pin):
        kw = dict(pin_memory=True) if pin else dict(device=dev)
        t = dict(n_kp=torch.zeros(n, dtype=torch.int32, **kw), n_det=torch.zeros(n, dtype=torch.int32, **kw),
                 uv_l=torch.zeros(n, cap, 2, **kw), uv_r=torch.zeros(n, cap, 2, **kw), xyz=torch.zeros(n, cap, 3, dtype=torch.float64, **kw),
                 dl=torch.zeros(n, cap, 32, dtype=torch.uint8, **kw), dr=torch.zeros(n, cap, 32, dtype=torch.uint8, **kw),
                 dist=torch.zeros(n, cap, dtype=torch.int32, **kw), idx=torch.zeros(n, cap, dtype=torch.int32, **kw),
                 st=torch.zeros(n, cap, dtype=torch.uint8, **kw))
        r = _lib.StereoResult(cap, t["n_kp"].data_ptr(), t["n_det"].data_ptr(), t["uv_l"].data_ptr(), t["uv_r"].data_ptr(), t["xyz"].data_ptr(),
                              t["dl"].data_ptr(), t["dr"].data_ptr(), t["dist"].data_ptr(), t["idx"].data_ptr(), t["st"].data_ptr())
        return t, r

    dout, dres = outputs(F, pin=False)
    stream = torch.cuda.current_stream().cuda_stream

    def device_step():
        fe.stereo_frames_device(dL.data_ptr(), dR.data_ptr(), W, W * H, F, dres, stream=stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (no profiling events inside the timed region)
    for _ in range(args.warmup):
        device_step()
    barrier()
    sampler = ClockSampler(dev_index)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        device_step()
    e1.record()
    barrier()
    clocks = sampler.stop()
    fe.check_overflow()   # the device-resident entry point reports candidate-list overflow here (never a silent cut)
    ms = e0.elapsed_time(e1)
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    total_frames = cfg["frames"] if cfg["scaling"] == "strong" else world * F
    value = total_frames * args.steps / (ms_max * 1e-3)
    if args.dump_outputs and rank == 0:   # before the profiled step below writes into the same buffers
        frames = dump_frame_sample(F, cap)
        sel = torch.as_tensor(frames, device=dev)
        write_stereo_dump(args.dump_outputs, {k: dout[v].index_select(0, sel).cpu().numpy() for k, v in RESULT_FIELDS.items()}, f_lo + frames)

    # ---- one extra step with every chunk on ONE stream: exclusive per-kernel durations for the roofline record
    fe.set_profiling(2)
    device_step()
    torch.cuda.synchronize()
    stages = fe.stage_timings()
    fe.set_profiling(0)

    if args.device_only:
        if rank == 0:
            print(json.dumps({"device_only": True, "config": args.config, "value": value, "ms_per_step": ms_max / args.steps, "clocks": clocks,
                              "stage_ms": {k: v["total_ms"] for k, v in stages.items()}}), flush=True)
        fe.close()
        return

    # ---- end to end through the host-buffer C-ABI call: pinned host in, pinned host out, every step.  Large batches go
    # through a pinned window of at most 4096 frames (the same number of bytes crosses the link per frame either way).
    Fh = min(F, 4096)
    hL = torch.empty((Fh, H, W), dtype=torch.uint8, pin_memory=True).copy_(dL[:Fh])
    hR = torch.empty((Fh, H, W), dtype=torch.uint8, pin_memory=True).copy_(dR[:Fh])
    ho, hres = outputs(Fh, pin=True)
    torch.cuda.synchronize()

    def host_step():
        done = 0
        while done < F:
            n = min(Fh, F - done)
            fe.stereo_frames_raw(hL.data_ptr(), hR.data_ptr(), W, W * H, n, hres)
            done += n

    for _ in range(max(1, args.warmup // 2)):
        host_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        host_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t_e = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = total_frames * args.steps / float(t_e.item())
    h2d = 2 * F * W * H
    d2h = F * cap * BYTES_PER_KEYPOINT + F * 8
    # what the host link can do on this box: one plain pinned -> device copy of the LEFT window, best of 3
    link_gbs = 0.0
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if hL.numel() >= (64 << 20):
        for _ in range(3):
            barrier()
            c0.record()
            dL[:Fh].copy_(hL, non_blocking=True)
            c1.record()
            torch.cuda.synchronize()
            link_gbs = max(link_gbs, hL.numel() / (c0.elapsed_time(c1) * 1e-3) / 1e9)

    # the two entry points must agree with each other (the host window holds frames 0 .. Fh-1)
    torch.cuda.synchronize()
    same = bool(torch.equal(dout["n_kp"][:Fh].cpu(), ho["n_kp"]))
    nk = ho["n_kp"].numpy()
    total_kp = int(nk.sum())
    total_ok = int((ho["st"].numpy() == 0)[np.arange(cap)[None, :] < nk[:, None]].sum())

    if rank == 0:
        chunk = fcfg["chunk_frames"]
        n_chunks = (F + chunk - 1) // chunk
        # kernels per chunk, from the library: harris_box, boxsum9, select_corners, the matcher, + describe_left on the
        # batch path, + bin_keypoints when the batch path bins the key-points (dense frames)
        per_chunk = kernels_per_chunk
        launches = args.steps * n_chunks * per_chunk
        peak, peak_src = measured_hbm_peak()
        ncu = ncu_kernel_metrics() if args.config == "c2" else {}
        sm_clk = (clocks.get("sm_mhz") or 1965) * 1e6
        roofline = None
        stages = {k: v for k, v in (stages or {}).items() if v["launches"]}
        if stages:
            frames_per_launch = min(chunk, F)
            tot_ms = sum(v["total_ms"] for v in stages.values())
            kernels = {}
            smem_peak = 148 * sm_clk   # one 128-byte wavefront of the L1 / shared data pipe per SM and clock
            for name, v in stages.items():
                avg = v["total_ms"] / v["launches"]
                rec = {"avg_launch_ms": avg, "share": v["total_ms"] / tot_ms, "hbm_gbs": frames_per_launch * frame_bytes / (avg * 1e-3) / 1e9}
                rec["hbm_frac"] = rec["hbm_gbs"] / peak
                if name in ncu:
                    rec["ncu"] = ncu[name]
                    wf = ncu[name].get("shared_wavefronts")
                    if wf and frames_per_launch == 64:   # the capture is a 64-frame launch of this configuration
                        rec["smem_wavefronts_per_s"] = wf / (avg * 1e-3)
                        rec["smem_frac"] = rec["smem_wavefronts_per_s"] / smem_peak
                kernels[name] = rec
            dom = max(kernels, key=lambda k: kernels[k]["avg_launch_ms"])
            k = kernels[dom]
            path_gbs = frame_bytes * (value / world) / 1e9
            # integer work of the matcher: 8 x 32-bit popc per candidate descriptor (SURVEY.md 8d), ~range candidates per key-point
            popc_per_frame = 8.0 * (total_kp / max(len(nk), 1)) * min(cfg.get("search_range", 60.0), W)
            popc_rate = (popc_per_frame * frames_per_launch / (kernels["stereo_match"]["avg_launch_ms"] * 1e-3)) if "stereo_match" in kernels else None
            popc_peak = 148 * 16 * sm_clk
            roofline = {"bound": "smem", "kernel": dom, "achieved": k["hbm_gbs"], "peak": peak, "unit": "GB/s", "frac": k["hbm_frac"],
                        "traffic": ncu.get(dom, {}).get("dram_bytes_per_launch"),
                        "peak_source": peak_src, "avg_launch_ms": k["avg_launch_ms"], "step_share": k["share"],
                        "frames_per_launch": frames_per_launch, "algorithmic_bytes_per_frame": frame_bytes,
                        "how": "one extra profiled step with all chunks on one stream: the library's CUDA events bracket exactly one kernel each",
                        "binding_unit": "shared-memory / L1 data pipe and instruction issue, not HBM (ncu: DRAM a few % of peak in every kernel; "
                                        "kernels[*].ncu, profiles/r2_*)",
                        "smem": {"achieved": k.get("smem_wavefronts_per_s"), "peak": smem_peak, "unit": "wavefronts/s", "frac": k.get("smem_frac"),
                                 "note": "LSU shared-memory wavefronts of one launch (ncu l1tex__data_pipe_lsu_wavefronts_mem_shared, committed capture) over "
                                         "the launch duration measured live, against 148 SMs x 1 wavefront per clock; TMA fills of the match windows "
                                         "use the same banks and are not in this count"},
                        "kernels": kernels,
                        "popc": {"per_s": popc_rate, "peak_per_s": popc_peak, "frac": (popc_rate / popc_peak) if popc_rate else None,
                                 "note": "XOR+popc of the Hamming distances in stereo_match (8 words per candidate) vs 148 SM x 16 lanes x SM clock; "
                                         "the kernel's time goes to the 256 BRIEF tests per candidate (shared-memory loads + packed compares)"},
                        "whole_path": {"achieved": path_gbs, "frac": path_gbs / peak,
                                       "note": "SURVEY.md 8d: B_frame x frames/s per GPU over the measured HBM peak"}}
        line = {
            "metric": metric_name(args.config, cams), "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": cfg["what"], "name": args.config, "frames_per_step_total": total_frames, "frames_this_rank": F,
                       "chunk_frames": chunk, "lanes": fcfg["n_lanes"], "device": dev_index, "cpu_affinity": args.numa,
                       "brief_table": fe.brief_table,
                       "l2_policy": (f"inputs {2 * F * W * H / 1e9:.2f} GB per step and rank >> 126 MB L2 (no flush needed)" if 2 * F * W * H > 4e8 else
                                     "the pair fits the L2: value = back-to-back calls on resident inputs; e2e brings new bytes from the host every call"),
                       "keypoints_per_frame": total_kp / max(len(nk), 1), "matched_per_frame": total_ok / max(len(nk), 1),
                       "device_vs_host_entry_equal": same},
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "h2d_gbs_achieved": h2d * args.steps / float(t_e.item()) / 1e9, "h2d_gbs_plain_copy": link_gbs or None,
                    "limiter": ("call latency" if F < 64 else "pcie_link" if world == 1 else "host_dram|pcie_switch (profiles/r2_h2d_matrix.json)"),
                    "note": "host link bound when h2d_gbs_achieved is close to h2d_gbs_plain_copy (rank 0's link)"},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
        }
        if world == 1 and not args.no_cpu_baseline:
            co, native = load_oracle()
            threads = co.host_threads()
            n_cpu = min(Fh, 4 * threads + 8)
            sl, sr = hL[:n_cpu].numpy(), hR[:n_cpu].numpy()
            fps_all, fps_one, n_s, ref = cpu_stereo_fps(co, native, oracle_config(co, cams, cfg), sl, sr, args.cpu_seconds, threads)
            got = {k: v.numpy() for k, v in ho.items()}
            ok = stereo_parity(ref, got, n_s)
            line["cpu_baseline"] = {"value": fps_all, "unit": "frames/s", "cores": threads, "kind": "port", "single_thread_value": fps_one,
                                    "sample": f"first {n_s} frames of the batch, {min(threads, n_s)} threads (one frame per thread), "
                                              f"{'-march=native' if native else 'x86-64-v3'} build of oracle/svi_oracle.c",
                                    "gpu_matches_cpu_on_sample": ok}
            line["gpu_matches_cpu_on_sample"] = ok
        print(json.dumps(line), flush=True)
    fe.close()


# ----------------------------------------------------------------------------- GPU arm: the tracking sequence (c3)
def cpp_tracker_timing(cfg, L, R, T):
    """The same sequence through the C++ host layer (svi_mapper_b200/host: CTrackerGT::process = trackManual + CLandmark
    optimisation + masked re-detection over the C-ABI) -- the reference-facing API a maintainer compiles into the tracker.
    Returns the demo driver's timing line, or why there is none."""
    import subprocess
    import tempfile

    import numpy as np
    exe = ROOT / "svi_mapper_b200" / "host" / "facade_demo"
    calib = ROOT / "tests" / "golden" / "calib"
    if not exe.exists():
        return {"unavailable": "svi_mapper_b200/host/facade_demo is not built"}
    n = len(L)
    with tempfile.TemporaryDirectory() as d:
        d = pathlib.Path(d)
        L.tofile(d / "L.raw")
        R.tofile(d / "R.raw")
        with open(d / "motions.txt", "w") as f:
            for t in range(n):
                M = np.eye(4) if t == 0 else T[t] @ np.linalg.inv(T[t - 1])
                a = float(np.arccos(np.clip((np.trace(M[:3, :3]) - 1.0) / 2.0, -1.0, 1.0)))
                f.write(" ".join(repr(float(v)) for v in M[:3].reshape(-1)) + " " + repr(a) + "\n")
        cmd = [str(exe), "--sequence", str(calib / f"{cfg['calib']}_left.txt"), str(calib / f"{cfg['calib']}_right.txt"), str(n),
               str(d / "L.raw"), str(d / "R.raw"), str(d / "motions.txt"), str(cfg["max_corners"]), str(d / "unused.txt")]
        best = None
        for _ in range(2):
            r = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, SVI_DEMO_TIMING="1"))
            if r.returncode != 0:
                return {"unavailable": (r.stderr or "facade_demo failed").strip()[-200:]}
            if os.environ.get("SVI_TRACE"):
                sys.stderr.write(r.stderr[-4000:])
            rec = json.loads(r.stdout.strip().splitlines()[-1])
            if best is None or rec["total_ms"] < best["total_ms"]:
                best = rec
    best["frames_per_s"] = best["frames"] / (best["total_ms"] * 1e-3)
    best["landmarks_per_s"] = best["landmarks_tracked"] / (best["total_ms"] * 1e-3)
    best["note"] = ("facade_demo --sequence (C++): wall time of CTrackerGT::process per frame after three warm-up frames, pageable images; "
                    "optimize_ms is optimizeActiveLandmarks = one svi_optimize_landmarks call per frame (CLandmark::optimize for every active landmark, "
                    "one warp each; a failed optimisation whose inputs did not change is repeated, not recomputed); 629 ms for the same 57 "
                    "frames with the host's per-landmark CPU loop (SVI_HOST_OPTIMIZE=cpu)")
    return best


def run_sequence(args, rank, world, dev_index):
    import numpy as np
    import torch
    import torch.distributed as dist

    from svi_mapper_b200 import StereoFrontend
    from svi_mapper_b200.sequence import GpuBackend, SequenceTracker, render_sequence

    cfg = args.cfg
    cams = cameras(cfg)
    W, H = cams[0].width, cams[0].height
    dev = torch.device("cuda", dev_index)
    n = cfg["frames"]
    L, R, T = render_sequence(cams[0], cams[1], n, cfg["seed"] + rank)   # every rank tracks its own replica of the workload
    # the tracker hands the library pinned frames (a camera driver's DMA buffers); results come back in host arrays
    pL = torch.empty((n, H, W), dtype=torch.uint8, pin_memory=True).copy_(torch.from_numpy(L))
    pR = torch.empty((n, H, W), dtype=torch.uint8, pin_memory=True).copy_(torch.from_numpy(R))
    Ln, Rn = pL.numpy(), pR.numpy()
    fe = StereoFrontend(cams[0], cams[1], device=dev_index, **frontend_kwargs(cfg))

    def one_pass():
        trk = SequenceTracker(GpuBackend(fe), cams[0])
        t_frames = []
        for t in range(n):
            t0 = time.perf_counter()
            trk.process(Ln[t], Rn[t], T[t])
            t_frames.append(time.perf_counter() - t0)
        return trk, t_frames

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(1, min(args.warmup, 2))):
        one_pass()
    barrier()
    sampler = ClockSampler(dev_index)
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        trk, t_frames = one_pass()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    t_e = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    dt_max = float(t_e.item())
    value = world * n * args.steps / dt_max
    if args.dump_outputs and rank == 0:
        write_sequence_dump(args.dump_outputs, trk)
    log = trk.log
    tracked = sum(r["tracked"] for r in log)
    stages = np.sum([r["stages"] for r in log], axis=0)
    # bytes of the calls of one sequence: two images up per frame; per tracked landmark 272 B up (xyz, two descriptors, disparity,
    # size, reference uv / descriptor / detection pose) and 106 B down (status, stage, two uv, xyz, two descriptors); a detection
    # frame adds 8 B per active landmark up (mask centres) and 113 B per key-point slot down
    lm_per_frame = tracked / n
    h2d = int(n * 2 * W * H + tracked * 272 + sum(r["active"] * 8 for r in log if r["new"]))
    d2h = int(tracked * 106 + sum(1 for r in log if r["new"]) * cfg["max_corners"] * BYTES_PER_KEYPOINT)
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        frame_bytes = 2 * W * H + lm_per_frame * (272 + 106)
        path_gbs = frame_bytes * (value / world) / 1e9
        track_ms = sorted(tf for tf, r in zip(t_frames, log) if not r["new"] and r["tracked"])
        detect_ms = sorted(tf for tf, r in zip(t_frames, log) if r["new"])
        line = {
            "metric": metric_name(args.config, cams), "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt_max / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": cfg["what"], "name": args.config, "frames_per_sequence": n, "landmarks_tracked_per_frame": lm_per_frame,
                       "landmarks_active_at_end": log[-1]["active"], "landmarks_per_s": world * tracked * args.steps / dt_max,
                       "stage_histogram": {"not_tracked": int(stages[0]), "stage1_left": int(stages[1]), "stage1_right": int(stages[2]),
                                           "stage2_left": int(stages[3]), "stage2_right": int(stages[4]), "stage3_epipolar": int(stages[5])},
                       "detections": sum(1 for r in log if r["new"]),
                       "ms_per_tracking_frame_median": (track_ms[len(track_ms) // 2] * 1e3) if track_ms else None,
                       "ms_per_detection_frame_median": (detect_ms[len(detect_ms) // 2] * 1e3) if detect_ms else None,
                       "replicas": "one independent sequence per rank (tracking does not shard inside a sequence: frame t needs the state of t-1)",
                       "l2_policy": "every frame arrives from pinned host memory (new images each call); nothing is reused across steps",
                       "value_is_e2e": "the tracker API is host-buffer based (svi_track_landmarks / svi_stereo_frame_masked): images go up and "
                                       "results come back inside every timed call, so value and e2e are the same measurement"},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "limiter": "call latency (one synchronous call per frame: ~10 small kernels + two copies + the Python bookkeeping)"},
            "gpu_launches": int(args.steps * sum(10 + (4 if r["new"] else 0) for r in log)), "clocks": clocks,
            "roofline": {"bound": "latency", "kernel": "track_stage1 / window detector / track_stage2 / track_stage3 (one call per frame)",
                         "achieved": path_gbs, "peak": peak, "unit": "GB/s", "frac": path_gbs / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_frame": frame_bytes,
                         "note": "a frame moves < 2 MB and launches kernels of a few thousand warps: the call is bound by launch + copy latency, "
                                 "neither by HBM nor by an execution pipe; ms_per_tracking_frame_median is the figure to compare"},
        }
        line["config"]["cpp_host"] = cpp_tracker_timing(cfg, L, R, T)
        if world == 1 and not args.no_cpu_baseline:
            co, native = load_oracle()
            threads = co.host_threads()
            ocfg = oracle_config(co, cams, cfg)
            # parity gate = the whole sequence in lockstep: GPU front-end and C port, state fed forward on both sides
            cpu = CpuSequenceBackend(co, native, ocfg, threads)
            g, c = SequenceTracker(GpuBackend(fe), cams[0]), SequenceTracker(cpu, cams[0])
            ok = True
            for t in range(n):
                rg, rc = g.process(Ln[t], Rn[t], T[t]), c.process(Ln[t], Rn[t], T[t])
                ok &= rg == rc
                if rg["tracked"] and ok:
                    a, b = g.last_track, c.last_track
                    hit = b["stage"] > 0
                    ok &= bool(np.array_equal(a["stage"], b["stage"]) and np.array_equal(a["status"], b["status"]))
                    ok &= all(bool(np.array_equal(a[k][hit], b[k][hit])) for k in ("uv_l", "uv_r", "desc_l", "desc_r"))
                    ok &= bool(np.allclose(a["xyz"][hit], b["xyz"][hit], rtol=1e-5, atol=0))
                ok = ok and all(bool(np.array_equal(g.s[k], c.s[k])) for k in g.s)
                if not ok:
                    break
            n_done = len(c.log)
            cpu_all = n_done / cpu.seconds
            lm_all = sum(r["tracked"] for r in c.log) / cpu.seconds
            # the reference walks the landmarks on ONE thread: time that on the first frames
            n1 = min(n, 12)
            cpu1 = CpuSequenceBackend(co, native, ocfg, 1)
            c1 = SequenceTracker(cpu1, cams[0])
            for t in range(n1):
                c1.process(Ln[t], Rn[t], T[t])
            line["cpu_baseline"] = {"value": cpu_all, "unit": "frames/s", "cores": threads, "kind": "port", "landmarks_per_s": lm_all,
                                    "single_thread_value": n1 / cpu1.seconds,
                                    "single_thread_landmarks_per_s": sum(r["tracked"] for r in c1.log) / cpu1.seconds,
                                    "sample": f"the whole {n}-frame sequence, landmark-parallel over {threads} threads (single thread: first {n1} frames), "
                                              f"{'-march=native' if native else 'x86-64-v3'} build of oracle/svi_oracle.c (C port of trackManual "
                                              f"+ addNewLandmarks)",
                                    "gpu_matches_cpu_on_sample": bool(ok)}
            line["gpu_matches_cpu_on_sample"] = bool(ok)
        print(json.dumps(line), flush=True)
    fe.close()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3  # timing rule: at least 3 warm-up steps

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU path")
    # Placement: on this pool's 8-GPU boxes GPUs 0-3 and 4-7 hang off two host uplinks of ~116 and ~142 GB/s
    # (profiles/r2_h2d_matrix.json: four neighbouring GPUs share 116 GB/s, four strided ones get 217 GB/s), so a job of
    # N < 8 ranks spreads its ranks over the visible devices (N=2 -> 0,4; N=4 -> 0,2,4,6) instead of packing them on 0..N-1.
    n_visible = torch.cuda.device_count()
    dev_index = local_rank * (n_visible // world) if (world <= n_visible and n_visible % world == 0) else local_rank % n_visible
    if args.device_order:
        order = [int(v) for v in args.device_order.split(",")]
        dev_index = order[local_rank % len(order)]
    torch.cuda.set_device(dev_index)
    # multi-GPU runs only: a single rank keeps every host core (its cpu_baseline leg uses them all)
    args.numa = bind_to_gpu_numa_node(dev_index) if (world > 1 and not args.no_numa_bind) else "all cpus"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev_index))
    try:
        if args.config == "c3":
            run_sequence(args, rank, world, dev_index)
        else:
            run_batch(args, rank, world, dev_index)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
