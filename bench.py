#!/usr/bin/env python3
"""bench.py — RGB-D frames/s of the PlanarSLAM per-frame hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one pass of the hot path over 7104 frames of a 256-frame synthetic 640x480 RGB-D sequence ("room corner", planarslam_b200/synth.py): four library
calls of 1776 frames for ORB / PEAC / PoseOptimization and two of 3552 for LSD, so that every call of a one-warp-per-frame kernel is exactly one resident wave.
With PSLAM_EXTRAS=1 (default) the extractors are followed by what the Frame constructor and Tracking run on their output: ComputeStereoFromRGBD, MatchORBPoints
against the previous frame, the key-frame exchange, LBD descriptors, isLineGood, the ComputePlanes post-processing, surface normals, TrackManhattanFrame.
Frames are independent units, so ranks shard them with no data-path collective (weak scaling: every rank processes FRAMES_PER_STEP frames per step); the
key-frame exchange is the one step that reads peer memory.  PSLAM_CONFIG=5 runs BASELINE.json's 1280x960 configuration.

Prints ONE JSON line on rank 0 (see DESIGN.md section 7 for every field):
  value      frames/s, inputs already resident in HBM, CUDA events on the launching stream, max over ranks
  e2e        frames/s through the host-pointer C ABI (pslam_frame_construct_batch + pslam_pose_optimization_batch): pinned H2D of the frames and D2H of
             every Frame product inside the timed region
  roofline   dominant kernel: algorithmic bytes per launch / its mean launch time (event-bracketed, measured live in a separate pass of the same
             workload) vs MEASURED_PEAKS.json hbm_gbs; per_kernel lists every kernel family
  cpu_baseline  the CPU path on the host cores: the reference's own code compiled here wherever it compiles, cv2 for the OpenCV calls, the oracle port for
             the rest (cpu_baseline.units says which); --impl reference prints the same thing as its own line
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# BASELINE.json configs: the default is configs[1] (640x480, 1000 ORB features), the configuration the metric is quoted on.  PSLAM_CONFIG=5 runs configs[4]
# (1280x960, 2000 features, frame-sharded with the peer-memory descriptor exchange) with the same step structure; it reports metric rgbd_frames_per_sec_1280x960.
CONFIG = os.environ.get("PSLAM_CONFIG", "2")
W, H = (1280, 960) if CONFIG == "5" else (640, 480)
NFEATURES = 2000 if CONFIG == "5" else 1000
AREA = (W * H) // (640 * 480)                                   # frames of config 5 carry 4x the pixels: per-frame byte counts and batch sizes scale with it
K_CAM = tuple(k * W / 640.0 for k in (535.4, 539.2, 320.1, 247.6))
# Frames per library call (context max_batch).  The serial-order kernels run one warp per frame, so throughput scales with
# frames in flight; the default is one full wave of the clustering kernel (pslam_peac_wave_frames: SMs x resident CTAs/SM,
# 1776 on a 148-SM B200), set in main().  1776 frames = 1.6 GB of gray+depth input >> 126 MB L2.
SUB_BATCH = int(os.environ.get("PSLAM_SUB_BATCH", "0"))
DEFAULT_WAVE = 1776 // min(AREA, 2)                                    # 148 SMs x 12 resident clustering CTAs (a quarter of a wave at 1280x960: device memory per frame is 4x)
SUBS_PER_STEP = int(os.environ.get("PSLAM_SUBS", "4"))         # ORB / PEAC / pose library calls per step (LSD takes the whole step in one call:
                                                               # its one-warp-per-frame kernel needs 32 frames per SM in flight, PEAC clustering fits 12)
FRAMES_PER_STEP = SUB_BATCH * SUBS_PER_STEP
LSD_SUBS = int(os.environ.get("PSLAM_LSD_SUBS", "2" if AREA == 1 else "4"))          # LSD calls per step: 4 x 1776 = 2 x 3552 frames, i.e. every LSD call is exactly one wave of its
                                                               # one-warp-per-frame kernel (24 resident CTAs per SM x 148), every PEAC call one wave of the clustering kernel (12 x 148)
DISTINCT_FRAMES = int(os.environ.get("PSLAM_DISTINCT_FRAMES", "256"))   # distinct frames of the replayed sequence (rendered on the host cores by a process pool)
                                                                         # and distinct pose problems; the step's frames cycle through them

# Algorithmic bytes per 640x480 frame of each kernel family (SURVEY.md §8d, restated in DESIGN.md §kernels)
ALGO_BYTES = {
    "orb_resize_level": 926546 + 850812,      # read levels 0-6 once, write levels 1-7 (borderless)
    "orb_fast_cells": 950532 + 30000 * 4,     # read every level once, write <= 30k packed candidates
    "orb_blur_level": 2 * 950532,             # read + write every level once
    "orb_blur_tma": 2 * 950532,               # same work, all levels in one TMA-staged launch
    "orb_quadtree": 30000 * 4 * 2,
    "orb_orient_describe": 1000 * (709 + 512 + 60),
    "peac_blocks": 614400 + 3072 * (17 * 8 + 5),       # read depth once, write per-block sums + PCA
    "peac_cluster": 2 * 3072 * (17 * 8 + 5) + 128 * 176,  # read block records, write node state + plane list
    "peac_seed": 1228800 + 1228800 + 8000 * 4,         # write labels + distance map + seed queue
    "peac_flood": 614400 + 130000 * (4 + 4 + 4 + 4),   # re-read depth at touched pixels, labels/dist RW, queue RW
    "peac_final_merge": 128 * 176 * 2,                 # coarse plane records in, final records out
    "peac_member_count": 1228800 + 300 * 128 * 4,      # labels read once, per-(sub-chunk, plane) counts written
    "peac_member_scan": 2 * 300 * 128 * 4,
    "peac_member_scatter": 2 * 1228800 + 1228800,      # labels read + rewritten, member index lists written
    "pose_optimization": 1046 * 104 + 1046 * 24 + 2048,   # edge records read once, residuals + flags written (per problem)
    "lsd_blur_scale": 307200 + 196608,                 # read the frame once, write the 512x384 scaled image
    "lsd_gradient": 196608 + 196608 * 16,              # read the scaled image, write one 16-byte record per pixel
    "lsd_regions": 196608 * 4 + 120000 * (4 + 8 + 4) + 60000 * 4 + 2 * 120000 * 4 + 2500 * 96,   # angle plane once, used-bit write + cos/sin + gradient of region pixels, seed order, region FIFO W+R, candidates
    "lsd_validate": 2500 * (96 + 8) + 2500 * 100 * 4,  # candidate rectangles + the angle words under each rectangle once
    "lsd_improve": 500 * (96 + 8) + 500 * 25 * 100 * 4,   # queued candidates: up to 25 more rectangle variants each
    "lsd_order": 2 * 196608 + 60000 * 4,               # the scaled image twice, the seed order once
    "lsd_emit": 2500 * 104 + 800 * 40,
    "lsd_keylines": 800 * 16 + 40 * (68 + 24),
    # chained extras
    "stereo_from_rgbd": 1000 * (28 + 2 + 8),           # key points + one depth sample each, uRight / depth out
    "hamming_knn2": 2 * 1000 * 32 + 1000 * 16,         # both descriptor sets once, two (index, distance) pairs per query
    "match_gate": 1000 * 12,
    "lbd_gradients": 307200 + 2 * 614400,              # the frame once, two int16 gradient planes
    "lbd_lines": 40 * 63 * 120 * 4 + 40 * 32,          # ~120 gradient samples on each of the 63 rows of a line's support region, 32 descriptor bytes
    "lines3d": 40 * (68 + 96) + 2040 * 2,              # key lines in, 3-D lines out, <= 51 depth samples per line
    "planes_post": 2 * 280000 * (4 + 2),               # member index + depth sample of every plane pixel, twice (bounding box, voxel pass)
    "planes_compact": 3 * 700 * 12 * 2,
    "sn_points": 34240 * (2 + 12), "sn_chamfer": 34240 * (12 + 1 + 4 * 3), "sn_gradients": 34240 * (12 + 24), "sn_integral": 34240 * 24 + 34615 * 48,
    "sn_normals": 34240 * (12 + 4 + 12) + 8 * 34615 * 24 // 4, "sn_gather": 8480 * (24 + 32 + 12),
    "exchange_publish": 2 * 1000 * (32 + 28), "exchange_match": 2 * 1000 * 32 + 1000 * 16,     # per key frame and peer record (8 key frames per step, not per frame)
    "track_manhattan": 8480 * 12 * 4 + 8480,           # the normals four times (cones, then one pass per axis), masks out
}
STAGES = [s for s in os.environ.get("PSLAM_STAGES", "orb,lsd,peac,pose").split(",") if s]
# the rest of the per-frame front end, chained on the stage that feeds it: ComputeStereoFromRGBD + MatchORBPoints after ORB, LBD descriptors + isLineGood after LSD,
# Frame::ComputePlanes' post-processing (voxel grid / RANSAC refit / surface normals) + TrackManhattanFrame after PEAC
EXTRAS = os.environ.get("PSLAM_EXTRAS", "1") != "0"


def _peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


DUMP_LIMIT = 64 << 20


def save_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32 (float32, and integers all below 2^24 in magnitude) or float64 (everything else), so every value
    stays exact; structured records become one column per scalar field.  Every written value is finite: where an output holds NaN or infinity (the
    direction of a rejected 3-D line, the normal of a pixel without depth), the value is written as 0 and out_dir/<name>_nonfinite.npy (float32, same
    shape) records 1 for NaN, 2 for +inf, 3 for -inf and 0 elsewhere.  Fails if the files would exceed DUMP_LIMIT bytes in all."""
    from numpy.lib import recfunctions
    conv = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype.names:
            a = recfunctions.structured_to_unstructured(a, dtype=np.float64)
        small_int = a.dtype.kind in "iub" and (a.size == 0 or int(np.abs(a.astype(np.int64)).max()) < (1 << 24))
        a = a.astype(np.float32 if a.dtype == np.float32 or small_int else np.float64)
        bad = ~np.isfinite(a)
        if bad.any():
            conv[name + "_nonfinite"] = np.select([np.isnan(a), a == np.inf, a == -np.inf], [1, 2, 3], 0).astype(np.float32)
            a = np.where(bad, 0, a).astype(a.dtype)
        conv[name] = a
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in conv.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


def make_frames(n_distinct=DISTINCT_FRAMES, world=1):
    from planarslam_b200 import synth
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    g, d = synth.render_sequence_parallel(seed=2, n=n_distinct, width=W, height=H, workers=max(1, min(64, cores // max(world, 1))))
    return g, d


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU every 100 ms while the timed region runs (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
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
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


CPU_UNITS = {}
CPU_SAMPLE_FRAMES = 16          # distinct rendered frames / pose problems the CPU arm cycles through


def _cpu_stage_fns(stages):
    """The per-frame CPU path, one callable per stage (called with a frame index), and what runs behind each.  ORB, PEAC and PoseOptimization are the
    reference's OWN code compiled unmodified in the build container (oracle/_ref/fast: src/ORBextractor.cc, src/PlaneExtractor.cpp + include/peac,
    src/Optimizer.cc + Thirdparty/g2o; -O3 -march=x86-64-v3, oracle/Makefile `fast`) where those libraries are present, else the oracle port; LSD is
    upstream OpenCV's own LineSegmentDetector (cv2, the implementation behind the reference's LSDDetector call) when cv2 imports, else the oracle port."""
    import oracle_lib
    import ref_lib
    from planarslam_b200 import synth_pose
    oracle_lib.lib()
    d = np.load(os.environ["PSLAM_CPU_FRAMES"])
    gray, depth = d["gray"], d["depth"]
    n = len(gray)
    probs = [synth_pose.make_pose_problem(11, frame=k) for k in range(n)]
    use_ref = os.environ.get("PSLAM_CPU_REF", "1") != "0"
    ref_orb = ref_lib.orb_lib() if use_ref else None
    ref_peac = ref_lib.peac_lib() if use_ref else None
    ref_match = ref_lib.match_lib() if use_ref else None
    lsd_cv = None
    if use_ref:
        try:
            import cv2
            cv2.setNumThreads(1)
            lsd_cv = cv2.createLineSegmentDetector(cv2.LSD_REFINE_ADV)
        except Exception:
            lsd_cv = None

    from planarslam_b200.lines import KEYLINE_DTYPE
    extras = EXTRAS
    cam = K_CAM
    depth_m = [(depth[k].astype(np.float32) * np.float32(1.0 / 5000.0)) for k in range(n)] if extras else None     # imDepth.convertTo(CV_32F, mDepthMapFactor): the caller's job
    bf = None
    if use_ref and extras:
        try:
            import cv2
            bf = cv2.BFMatcher(cv2.NORM_HAMMING)
        except Exception:
            bf = None
    prev_desc = {}

    def keylines_of(segs):
        """KeyLines of ExtractLineSegment (LSDDetector::detect fields used downstream) from cv2's segments: 40 longest, end points clamped into the image."""
        kl = np.zeros(len(segs), KEYLINE_DTYPE)
        if len(segs):
            sx, sy = np.clip(segs[:, 0], 0, W - 1), np.clip(segs[:, 1], 0, H - 1)
            ex, ey = np.clip(segs[:, 2], 0, W - 1), np.clip(segs[:, 3], 0, H - 1)
            kl["startPointX"], kl["startPointY"], kl["endPointX"], kl["endPointY"] = sx, sy, ex, ey
            kl["sPointInOctaveX"], kl["sPointInOctaveY"], kl["ePointInOctaveX"], kl["ePointInOctaveY"] = sx, sy, ex, ey
            kl["lineLength"] = np.hypot(ex - sx, ey - sy)
            kl["angle"] = np.arctan2(ey - sy, ex - sx)
            kl["pt"][:, 0], kl["pt"][:, 1] = (sx + ex) / 2, (sy + ey) / 2
            kl["size"] = np.abs(ex - sx) * np.abs(ey - sy)
            kl["class_id"] = np.arange(len(segs))
            kl["numOfPixels"] = np.maximum(np.abs(ex - sx), np.abs(ey - sy)).astype(np.int32) + 1
        return kl

    def f_lsd(i):
        g = gray[i % n]
        if lsd_cv is None:
            kl = oracle_lib.extract_line_segments(g, 40)
            kl = kl[0] if isinstance(kl, tuple) else kl
        else:
            segs = lsd_cv.detect(g)[0]                       # + ExtractLineSegment's keep-40 (src/LSDextractor.cpp:18-26)
            segs = segs.reshape(-1, 4) if segs is not None else np.zeros((0, 4), np.float32)
            segs = segs[np.argsort(-np.hypot(segs[:, 2] - segs[:, 0], segs[:, 3] - segs[:, 1]), kind="stable")[:40]]
            kl = keylines_of(segs) if extras else None
        if extras:
            oracle_lib.lbd_compute(g, kl)                                                      # BinaryDescriptor::compute (port: opencv_contrib is not in this image)
            (ref_lib.ref_full_lines3d_frame if ref_match else oracle_lib.lines3d_frame)(kl, depth_m[i % n], cam, 1)        # Frame::isLineGood

    def f_orb(i):
        g = gray[i % n]
        r = ref_lib.ref_orb_extract(g, nfeatures=NFEATURES, monotonic_alloc=False) if ref_orb else oracle_lib.orb_extract(g, nfeatures=NFEATURES)
        if extras:
            kps, desc = r[0], r[1]
            xy = np.ascontiguousarray(np.stack([kps["x"], kps["y"]], 1), np.float32)
            (ref_lib.ref_full_compute_stereo_from_rgbd if ref_match else oracle_lib.compute_stereo_from_rgbd)(xy, xy, depth_m[i % n], 40.0)
            last = prev_desc.get("d")
            if last is not None and len(last) and len(desc):                                   # MatchORBPoints against the previous frame of this worker
                if bf is not None:
                    m = bf.match(np.ascontiguousarray(desc), last)
                    dmin = min((x.distance for x in m), default=0.0)
                    [x for x in m if x.distance <= max(2 * dmin, 30.0)]
                else:
                    xor = np.bitwise_xor(np.ascontiguousarray(desc)[:, None, :], last[None, :, :])
                    np.unpackbits(xor, axis=2).sum(2).argmin(1)
            prev_desc["d"] = np.ascontiguousarray(desc)

    R_eye = np.eye(3, dtype=np.float32)
    ref_track = ref_lib.track_lib() if (use_ref and extras) else None

    def f_peac(i):
        d = depth[i % n]
        if not extras:
            return ref_lib.ref_peac_time(d, K=K_CAM) if ref_peac else oracle_lib.PeacOracle(d, K=K_CAM)
        # Frame::ComputePlanes: PEAC + the per-plane post-processing + surface normals, then TrackManhattanFrame on the normals.  The post-processing consumes
        # the PEAC result in memory, so the whole function runs in the port here (one PEAC pass, not the compiled reference's plus the port's)
        oracle_lib.planes_post(d, K=K_CAM)
        sn = oracle_lib.surface_normals(d, K=K_CAM)
        nr = np.ascontiguousarray(sn[:, :3])
        (ref_lib.ref_track_manhattan_frame if ref_track else oracle_lib.track_manhattan_frame)(R_eye, nr, np.zeros((0, 3)))

    fns = {"orb": f_orb, "lsd": f_lsd, "peac": f_peac,
           "pose": (lambda i: ref_lib.ref_full_pose_optimization(probs[i % n], False)) if ref_match else (lambda i: oracle_lib.pose_optimization(probs[i % n]))}
    units = {"orb": "reference src/ORBextractor.cc (OpenCV primitives inside it: scalar restatements)" if ref_orb else "port",
             "lsd": "upstream cv2 LineSegmentDetector (1 thread)" if lsd_cv is not None else "port",
             "peac": ("reference src/PlaneExtractor.cpp + include/peac" if ref_peac else "port") if not extras else
                     "port of the whole Frame::ComputePlanes (PEAC + VoxelGrid / RANSAC refit + surface normals; PCL is not in this image)",
             "pose": "reference src/Optimizer.cc PoseOptimization(Frame*) + Thirdparty/g2o" if ref_match else "port"}
    if extras:
        units["orb"] += " + Frame::ComputeStereoFromRGBD (compiled src/Frame.cc) + cv2.BFMatcher (MatchORBPoints)" if (ref_match and bf is not None) else " + stereo / matching ports"
        units["lsd"] += " + LBD port + Frame::isLineGood (compiled src/Frame.cc)" if ref_match else " + LBD / isLineGood ports"
        units["peac"] += " + Tracking::TrackManhattanFrame (compiled src/Tracking.cc)" if ref_track else " + Manhattan port"
    return {k: v for k, v in fns.items() if k in stages}, {k: v for k, v in units.items() if k in stages}


def cpu_worker_main(spec):
    """Child process of the CPU arm (python bench.py --cpu-worker '<json>'): pinned to one core (or three for the reference's thread-per-extractor
    mode), prints 'ready <units json>', then for every line 'go <first frame> <count>' on stdin processes the frames and prints 'done <seconds>'."""
    os.environ["PSLAM_REF_VARIANT"] = "fast"
    cores = spec["cores"]
    try:
        os.sched_setaffinity(0, set(cores))
    except Exception:
        pass
    fns, units = _cpu_stage_fns(spec["stages"])
    par = [k for k in ("orb", "lsd", "peac") if k in fns]
    pool = None
    if spec["mode"] == "ref3":
        from concurrent.futures import ThreadPoolExecutor
        pool = ThreadPoolExecutor(3)

    def frame(i):
        if pool is not None:                       # Frame::Frame: three std::threads (ExtractORB, ExtractLSD, ComputePlanes), join, src/Frame.cc:90-95
            for f in [pool.submit(fns[k], i) for k in par]:
                f.result()
        else:
            for k in par:
                fns[k](i)
        if "pose" in fns:
            fns["pose"](i)

    frame(spec["rank"])                            # warm (page in the libraries, the frames)
    sys.stdout.write("ready " + json.dumps(units) + "\n")
    sys.stdout.flush()
    for line in sys.stdin:
        tok = line.split()
        if not tok or tok[0] != "go":
            break
        first, count = int(tok[1]), int(tok[2])
        t0 = time.perf_counter()
        for i in range(first, first + count):
            frame(i)
        sys.stdout.write(f"done {time.perf_counter() - t0:.6f}\n")
        sys.stdout.flush()


class CpuArm:
    """Process pool of pinned CPU workers (one Python process per core, or per three cores in 'ref3' mode); a step = every worker processes
    `per_worker` frames between a common start signal and the last 'done'."""

    def __init__(self, gray, depth, mode, n_workers, stages):
        import subprocess
        import tempfile
        self.mode, self.n = mode, n_workers
        self.tmp = tempfile.NamedTemporaryFile(suffix=".npz", delete=False)
        np.savez(self.tmp, gray=gray, depth=depth)
        self.tmp.close()
        avail = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
        width = 3 if mode == "ref3" else 1
        env = dict(os.environ, PSLAM_CPU_FRAMES=self.tmp.name, PSLAM_REF_VARIANT="fast", OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1",
                   CUDA_VISIBLE_DEVICES="")
        self.procs = []
        for r in range(n_workers):
            spec = {"mode": mode, "rank": r, "stages": stages, "cores": [avail[(r * width + k) % len(avail)] for k in range(width)]}
            self.procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cpu-worker", json.dumps(spec)], stdin=subprocess.PIPE,
                                               stdout=subprocess.PIPE, text=True, env=env))
        self.units = {}
        for p in self.procs:
            line = p.stdout.readline()
            if not line.startswith("ready"):
                raise RuntimeError("CPU worker failed to start: " + line)
            self.units = json.loads(line[6:])

    def step(self, per_worker):
        t0 = time.perf_counter()
        for r, p in enumerate(self.procs):
            p.stdin.write(f"go {r * per_worker} {per_worker}\n")
            p.stdin.flush()
        for p in self.procs:
            line = p.stdout.readline()
            if not line.startswith("done"):
                raise RuntimeError("CPU worker died: " + line)
        return time.perf_counter() - t0, per_worker * self.n

    def close(self):
        for p in self.procs:
            try:
                p.stdin.close()
                p.wait(timeout=10)
            except Exception:
                p.kill()
        try:
            os.unlink(self.tmp.name)
        except OSError:
            pass


def cpu_modes(gray, depth, seconds=8.0):
    """BASELINE.md section 3's three threading modes of the CPU path on this box: one thread; the reference's own layout (three extractor threads per
    frame, src/Frame.cc:90-95, one frame at a time per process) replicated over cores // 3 processes; one frame per core on all cores."""
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    out = {}
    for name, mode, nw in (("single_thread", "seq", 1), ("three_threads_per_frame", "ref3", max(1, cores // 3)), ("frame_parallel_all_cores", "seq", cores)):
        arm = CpuArm(gray, depth, mode, nw, STAGES)
        try:
            arm.step(1)
            t, n = 0.0, 0
            while t < seconds:
                dt, k = arm.step(2)
                t += dt
                n += k
            out[name] = {"frames_per_sec": round(n / t, 3), "processes": nw, "threads": nw * (3 if mode == "ref3" else 1), "frames": n, "seconds": round(t, 2)}
            CPU_UNITS.clear()
            CPU_UNITS.update(arm.units)
        finally:
            arm.close()
    out["host_cores"] = cores
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path on all host cores of this box (rank 0 only): one pinned worker process per core, each running whole
    frames through ORB + LSD + PEAC + PoseOptimization (see _cpu_stage_fns for what code runs behind each stage).  A step = 4 frames per worker; ms_per_step
    is that step's measured wall time, value = frames of the timed steps / their summed time."""
    if rank != 0:
        return
    global SUB_BATCH, FRAMES_PER_STEP
    if SUB_BATCH <= 0:
        SUB_BATCH = DEFAULT_WAVE
    gray, depth = make_frames(CPU_SAMPLE_FRAMES)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per_worker = int(os.environ.get("PSLAM_CPU_FRAMES_PER_WORKER", "4"))
    arm = CpuArm(gray, depth, "seq", cores, STAGES)
    try:
        for _ in range(max(args.warmup, 0)):
            arm.step(per_worker)
        tot_t, tot_n = 0.0, 0
        for _ in range(max(args.steps, 1)):
            dt, n = arm.step(per_worker)
            tot_t += dt
            tot_n += n
        units = dict(arm.units)
    finally:
        arm.close()
    FRAMES_PER_STEP = per_worker * cores
    v = tot_n / tot_t
    cfg = workload_config()
    cfg["reference_step"] = f"{per_worker} frames on each of {cores} pinned worker processes ({FRAMES_PER_STEP} frames per step, {CPU_SAMPLE_FRAMES} distinct)"
    line = {"impl": "reference", "metric": f"rgbd_frames_per_sec_{W}x{H}", "value": v, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * tot_t / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "reference", "units": units,
                             "sample": f"{' + '.join(STAGES)}: {tot_n} frames in {tot_t:.1f} s, one pinned process per core ({cores}), -O3 -march=x86-64-v3"},
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config():
    return {"workload": f"{W}x{H} synthetic RGB-D sequence: ORB ({NFEATURES} feats, 8 levels) + LSD line segments (REFINE_ADV, 40 longest -> KeyLines + "
                        "line functions) + PEAC planes + PoseOptimization (1000 point + 40 line (80 edges) + 6 plane "
                        "edges per frame)",
            "frames_per_step": FRAMES_PER_STEP, "sub_batch": SUB_BATCH, "distinct_frames": DISTINCT_FRAMES, "l2": "inputs_larger_than_l2",
            "stages": STAGES, "streams": len(STAGES),
            "extras": ("ComputeStereoFromRGBD + MatchORBPoints (consecutive frames) after ORB; LBD descriptors + isLineGood after LSD; ComputePlanes post-processing "
                       "(VoxelGrid, RANSAC refit, surface normals) + TrackManhattanFrame (surface normals only) after PEAC") if EXTRAS else "off"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (a fixed sample of frames; rank 0)")
    ap.add_argument("--cpu-worker", default=None, help=argparse.SUPPRESS)       # internal: child process of the CPU arm
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    if args.cpu_worker:
        cpu_worker_main(json.loads(args.cpu_worker))
        return

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from planarslam_b200._lib import Context, KEYPOINT_DTYPE, PLANE_DTYPE
    from planarslam_b200.optimizer import Optimizer
    from planarslam_b200 import synth_pose

    global SUB_BATCH, FRAMES_PER_STEP
    if SUB_BATCH <= 0:
        probe = Context(W, H, 1, device=local_rank)
        SUB_BATCH = (int(probe.L.pslam_peac_wave_frames(probe.h)) or 1776) // min(AREA, 2)          # config 5: half a wave per call (device memory per frame is 4x)
        del probe
    FRAMES_PER_STEP = SUB_BATCH * SUBS_PER_STEP
    assert LSD_SUBS <= SUBS_PER_STEP

    gray, depth = make_frames(world=world)
    if world > 1:          # every rank replays the sequence from a different position, so that the key frames the ranks exchange differ
        shift = rank * (len(gray) // world)
        gray, depth = np.roll(gray, -shift, axis=0), np.roll(depth, -shift, axis=0)
    # the step's frames are built once, directly in page-locked host memory (the buffers the end-to-end leg hands to the ABI): the DISTINCT_FRAMES
    # frames of the rendered sequence, repeated in order until the step is full
    h_gray = torch.empty((FRAMES_PER_STEP, H, W), dtype=torch.uint8).pin_memory()
    h_depth = torch.empty((FRAMES_PER_STEP, H, W), dtype=torch.int16).pin_memory()      # uint16 bits
    hg, hd = h_gray.numpy(), h_depth.numpy()
    for o in range(0, FRAMES_PER_STEP, DISTINCT_FRAMES):
        n = min(DISTINCT_FRAMES, FRAMES_PER_STEP - o)
        hg[o:o + n] = gray[:n]
        hd[o:o + n] = depth[:n].view(np.int16)
    dev = torch.device("cuda", local_rank)
    main = torch.cuda.current_stream(dev)
    # ORB, PEAC, pose.  The PEAC chain (one warp per frame, latency-bound) is the critical path: high priority, so its CTAs
    # are placed first and the bulk-parallel ORB / pose kernels fill the remaining issue slots.
    streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev, priority=-1), torch.cuda.Stream(dev), torch.cuda.Stream(dev, priority=-1)]
    ctxs = [Context(W, H, SUB_BATCH, device=local_rank, nfeatures=NFEATURES) for _ in range(3)] + [Context(W, H, (FRAMES_PER_STEP + LSD_SUBS - 1) // LSD_SUBS, device=local_rank)]   # one context per stage family
    # PSLAM_LSD_STREAM=peac puts the two latency-bound one-warp-per-frame chains (PEAC, LSD) on one stream: their CTAs compete for
    # the same register file, and running them back to back avoids half-resident waves of both
    # (config 5: a call holds a quarter of the frames the one-warp-per-frame kernels could keep resident, so the two chains overlap on separate streams)
    mode = os.environ.get("PSLAM_LSD_STREAM", "peac" if AREA == 1 else "own")
    if mode == "peac":
        streams[3] = streams[1]
    elif mode == "one":
        streams[0] = streams[2] = streams[3] = streams[1]
    elif mode == "two":                     # bulk-parallel families (ORB, pose) on one stream, serial-order families (PEAC, LSD) on the other
        streams[2] = streams[0]
        streams[3] = streams[1]
    for c, st in zip(ctxs, streams):
        c.set_stream(st.cuda_stream)
    c_orb, c_peac, c_pose, c_lsd = ctxs
    from planarslam_b200.lines import KEYLINE_DTYPE
    MAX_LINES = 40
    cap = c_orb.L.pslam_orb_max_keypoints(c_orb.h)
    maxp = c_peac.L.pslam_peac_max_planes(c_peac.h)
    L = c_orb.L

    d_gray = h_gray.to(dev)                                            # [FRAMES_PER_STEP, H, W] resident in HBM
    d_depth = h_depth.to(dev)
    d_kps = torch.empty((SUB_BATCH, cap, 28), dtype=torch.uint8, device=dev)
    d_desc = torch.empty((SUB_BATCH, cap, 32), dtype=torch.uint8, device=dev)
    d_n = torch.zeros(FRAMES_PER_STEP, dtype=torch.int32, device=dev)
    d_labels = torch.empty((SUB_BATCH, H * W), dtype=torch.int32, device=dev)
    d_planes = torch.empty((SUB_BATCH, maxp, PLANE_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    d_npl = torch.zeros(FRAMES_PER_STEP, dtype=torch.int32, device=dev)
    d_members = torch.empty((SUB_BATCH, H * W), dtype=torch.int32, device=dev)
    d_moff = torch.empty((SUB_BATCH, maxp + 1), dtype=torch.int32, device=dev)
    d_kl = torch.empty((FRAMES_PER_STEP, MAX_LINES, KEYLINE_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    d_lf = torch.empty((FRAMES_PER_STEP, MAX_LINES, 3), dtype=torch.float64, device=dev)
    d_nkl = torch.zeros(FRAMES_PER_STEP, dtype=torch.int32, device=dev)
    def pinned(shape, dtype):          # page-locked host result buffers (what a replay driver would hand to the ABI)
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        t = torch.empty(n, dtype=torch.uint8).pin_memory()
        pinned.keep.append(t)
        return t.numpy().view(dtype).reshape(shape)
    pinned.keep = []
    h_kps = pinned((SUB_BATCH, cap), KEYPOINT_DTYPE)
    h_desc = pinned((SUB_BATCH, cap, 32), np.uint8)
    h_n = pinned((SUB_BATCH,), np.int32)
    h_labels = pinned((SUB_BATCH, H * W), np.int32)
    h_planes = pinned((SUB_BATCH, maxp), PLANE_DTYPE)
    h_npl = pinned((SUB_BATCH,), np.int32)
    h_kl = pinned((FRAMES_PER_STEP, MAX_LINES), KEYLINE_DTYPE)
    h_lf = pinned((FRAMES_PER_STEP, MAX_LINES, 3), np.float64)
    h_nkl = pinned((FRAMES_PER_STEP,), np.int32)
    # pose problems: one per frame of a sub-batch (the correspondences a tracker would hand over), packed + uploaded once
    base_probs = [synth_pose.make_pose_problem(11 + k // 64, frame=k % 64) for k in range(DISTINCT_FRAMES)]
    probs = [base_probs[k % DISTINCT_FRAMES] for k in range(SUB_BATCH)]
    opt = Optimizer(c_pose)
    opt.pack(probs)
    pose_h2d = sum(sum(p[k].nbytes for k in ("Xw", "obs", "inv_sigma2", "line_Xw", "line_obs", "plane_meas", "plane_map", "par_meas",
                                              "par_map", "ver_meas", "ver_map")) + 64 for p in probs)

    # ---- buffers of the chained extras ----
    h_ur, h_dz = pinned((SUB_BATCH, cap), np.float32), pinned((SUB_BATCH, cap), np.float32)
    h_ldesc = pinned((FRAMES_PER_STEP, MAX_LINES, 32), np.uint8)
    h_l3d = pinned((FRAMES_PER_STEP, MAX_LINES, 96), np.uint8)
    h_seed, h_drawn = pinned((FRAMES_PER_STEP,), np.uint32), pinned((FRAMES_PER_STEP,), np.int32)
    h_seed[:] = 1
    h_pp_n, h_pp_src, h_pp_coef = pinned((SUB_BATCH,), np.int32), pinned((SUB_BATCH, maxp), np.int32), pinned((SUB_BATCH, maxp, 4), np.float32)
    h_pp_off, h_pp_pts = pinned((SUB_BATCH, maxp + 1), np.int32), pinned((SUB_BATCH, 4096, 3), np.float32)
    h_sn8 = pinned((SUB_BATCH, int(L.pslam_surface_normals_count(c_peac.h)), 8), np.float32)
    L.pslam_compute_stereo_from_rgbd_batch.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    L.pslam_compute_planes_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p]
    L.pslam_lines_extract_describe_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 5
    L.pslam_lines3d_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_float] + [C.c_void_p] * 5
    from planarslam_b200.lines import LINE3D_DTYPE
    from planarslam_b200.manhattan import MANHATTAN_RESULT_DTYPE
    DEPTH_FACTOR, BF, DIST_TH = float(np.float32(1.0 / 5000.0)), 40.0, 0.05
    cam4 = (C.c_float * 4)(*K_CAM)
    n_sn = int(L.pslam_surface_normals_count(c_peac.h))
    PP_CAP = 4096
    d_ur = torch.empty((SUB_BATCH, cap), dtype=torch.float32, device=dev); d_dz = torch.empty_like(d_ur)
    d_midx = torch.empty((SUB_BATCH, cap, 2), dtype=torch.int32, device=dev); d_mdist = torch.empty_like(d_midx)
    d_good = torch.empty((SUB_BATCH, cap), dtype=torch.int32, device=dev); d_ngood = torch.zeros(SUB_BATCH, dtype=torch.int32, device=dev)
    d_ldesc = torch.empty((FRAMES_PER_STEP, MAX_LINES, 32), dtype=torch.uint8, device=dev)
    d_l3d = torch.empty((FRAMES_PER_STEP, MAX_LINES, LINE3D_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    d_seed = torch.ones(FRAMES_PER_STEP, dtype=torch.int32, device=dev); d_drawn = torch.zeros(FRAMES_PER_STEP, dtype=torch.int32, device=dev)
    d_pp_n = torch.zeros(SUB_BATCH, dtype=torch.int32, device=dev); d_pp_src = torch.empty((SUB_BATCH, maxp), dtype=torch.int32, device=dev)
    d_pp_coef = torch.empty((SUB_BATCH, maxp, 4), dtype=torch.float32, device=dev); d_pp_off = torch.empty((SUB_BATCH, maxp + 1), dtype=torch.int32, device=dev)
    d_pp_pts = torch.empty((SUB_BATCH, PP_CAP, 3), dtype=torch.float32, device=dev); d_pp_status = torch.zeros(SUB_BATCH, dtype=torch.int32, device=dev)
    d_sn8 = torch.empty((SUB_BATCH, n_sn, 8), dtype=torch.float32, device=dev); d_sn3 = torch.empty((SUB_BATCH, n_sn, 3), dtype=torch.float32, device=dev)
    d_nsn = torch.full((SUB_BATCH,), n_sn, dtype=torch.int32, device=dev); d_ndirs = torch.zeros(SUB_BATCH, dtype=torch.int32, device=dev)
    d_dirs = torch.zeros((SUB_BATCH, 1, 3), dtype=torch.float64, device=dev)
    d_Rlast = torch.eye(3, dtype=torch.float32, device=dev).repeat(SUB_BATCH, 1, 1).contiguous()
    d_mres = torch.empty((SUB_BATCH, MANHATTAN_RESULT_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    d_nmask = torch.empty((SUB_BATCH, n_sn), dtype=torch.uint8, device=dev); d_dmask = torch.empty((SUB_BATCH, 1), dtype=torch.uint8, device=dev)
    L.pslam_compute_stereo_from_rgbd_batch_dev.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    L.pslam_lines_extract_describe_batch_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 4
    L.pslam_lines3d_batch_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_float] + [C.c_void_p] * 5
    L.pslam_planes_post_batch_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_float] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p]
    L.pslam_surface_normals_batch_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.pslam_track_manhattan_batch_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]

    # key-frame exchange (SURVEY.md section 8e): every step, each rank publishes the ORB blocks of KF of its frames into records in its own HBM and matches
    # them against the records of ALL ranks read in place over NVLink (one fused wait-on-flag + Hamming k = 2 kernel per key frame); two slot sets alternate
    # by epoch parity, so a slot is rewritten only after every peer has matched it (publish(e + 2) is stream-ordered after this rank's match(e + 1), which
    # waited for every peer's publish(e + 1), itself stream-ordered after that peer's match(e))
    KF = int(os.environ.get("PSLAM_KEYFRAMES_PER_STEP", "8"))
    xch, xch_epoch = None, [0]
    if EXTRAS and "orb" in STAGES and KF > 0:
        from planarslam_b200.sharding import PeerDescriptorExchange
        xch = PeerDescriptorExchange(c_orb, cap, slots=2 * KF)
        d_xidx = torch.empty((KF, cap, 2), dtype=torch.int32, device=dev); d_xdist = torch.empty_like(d_xidx)
        kf_stride = max(SUB_BATCH // KF, 1)

    def dev_orb(o):
        c_orb.check(L.pslam_orb_extract_batch_dev(c_orb.h, d_gray[o].data_ptr(), SUB_BATCH, d_kps.data_ptr(), d_desc.data_ptr(), cap,
                                                  d_n[o:].data_ptr()))
        if EXTRAS:
            c_orb.check(L.pslam_compute_stereo_from_rgbd_batch_dev(c_orb.h, d_kps.data_ptr(), d_kps.data_ptr(), d_n[o:].data_ptr(), cap, d_depth[o].data_ptr(), SUB_BATCH,
                                                                   DEPTH_FACTOR, BF, d_ur.data_ptr(), d_dz.data_ptr()))
            # MatchORBPoints of every frame against its predecessor in the sub-batch (cv::BFMatcher 1-NN + the 2 x min-distance gate)
            c_orb.check(L.pslam_hamming_knn2_batch_dev(c_orb.h, d_desc[1:].data_ptr(), d_n[o + 1:].data_ptr(), cap, d_desc.data_ptr(), d_n[o:].data_ptr(), cap,
                                                       SUB_BATCH - 1, d_midx.data_ptr(), d_mdist.data_ptr(), d_good.data_ptr(), d_ngood.data_ptr()))
            if xch is not None and o == 0:
                xch_epoch[0] += 1
                e, base = xch_epoch[0], (xch_epoch[0] & 1) * KF
                for k in range(KF):
                    f = min(k * kf_stride, SUB_BATCH - 1)
                    xch.publish(base + k, d_desc[f], d_n[f:f + 1], e, d_kps[f])
                for k in range(KF):
                    f = min(k * kf_stride, SUB_BATCH - 1)
                    xch.match(base + k, e, d_desc[f], d_n[f:f + 1], d_xidx[k], d_xdist[k])

    def dev_peac(o):
        c_peac.check(L.pslam_peac_run_batch_dev(c_peac.h, d_depth[o].data_ptr(), SUB_BATCH, d_labels.data_ptr(), d_planes.data_ptr(),
                                                d_npl[o:].data_ptr(), d_members.data_ptr(), d_moff.data_ptr()))
        if EXTRAS:
            c_peac.check(L.pslam_planes_post_batch_dev(c_peac.h, d_depth[o].data_ptr(), SUB_BATCH, d_planes.data_ptr(), d_npl[o:].data_ptr(), d_members.data_ptr(),
                                                       d_moff.data_ptr(), DIST_TH, d_pp_n.data_ptr(), d_pp_src.data_ptr(), d_pp_coef.data_ptr(), d_pp_off.data_ptr(),
                                                       d_pp_pts.data_ptr(), PP_CAP, d_pp_status.data_ptr()))
            c_peac.check(L.pslam_surface_normals_batch_dev(c_peac.h, d_depth[o].data_ptr(), SUB_BATCH, d_sn8.data_ptr(), d_sn3.data_ptr()))
            c_peac.check(L.pslam_track_manhattan_batch_dev(c_peac.h, d_Rlast.data_ptr(), d_sn3.data_ptr(), d_nsn.data_ptr(), n_sn, d_dirs.data_ptr(), d_ndirs.data_ptr(), 1,
                                                           SUB_BATCH, d_mres.data_ptr(), d_nmask.data_ptr(), d_dmask.data_ptr()))

    LSD_BATCH = (FRAMES_PER_STEP + LSD_SUBS - 1) // LSD_SUBS

    def dev_lsd(j=None):
        for q in (range(LSD_SUBS) if j is None else [j]):
            o, n = q * LSD_BATCH, min(LSD_BATCH, FRAMES_PER_STEP - q * LSD_BATCH)
            if EXTRAS:
                c_lsd.check(L.pslam_lines_extract_describe_batch_dev(c_lsd.h, d_gray[o].data_ptr(), n, MAX_LINES, d_kl[o].data_ptr(), d_lf[o].data_ptr(),
                                                                     d_ldesc[o].data_ptr(), d_nkl[o:].data_ptr()))
                c_lsd.check(L.pslam_lines3d_batch_dev(c_lsd.h, d_kl[o].data_ptr(), d_nkl[o:].data_ptr(), MAX_LINES, d_depth[o].data_ptr(), n, DEPTH_FACTOR, cam4,
                                                      d_seed[o:].data_ptr(), None, d_l3d[o].data_ptr(), d_drawn[o:].data_ptr()))
            else:
                c_lsd.check(L.pslam_lines_extract_batch_dev(c_lsd.h, d_gray[o].data_ptr(), n, MAX_LINES, d_kl[o].data_ptr(), d_lf[o].data_ptr(),
                                                            d_nkl[o:].data_ptr()))

    def steps_dev(nsteps):
        """nsteps passes over the batch.  The three stage families are independent per frame, so each runs its own
        sequence of batches on its stream (fork at the start, join at the end: ORB of pass i+1 may overlap PEAC of pass i)."""
        ev = torch.cuda.Event()
        ev.record(main)
        for st in streams:
            st.wait_event(ev)
        for _ in range(nsteps):
            for s in range(SUBS_PER_STEP):
                o = s * SUB_BATCH
                if "lsd" in STAGES and s < LSD_SUBS:
                    dev_lsd(s)
                if "peac" in STAGES:
                    dev_peac(o)
                if "orb" in STAGES:
                    dev_orb(o)
                if "pose" in STAGES:
                    opt.run_packed()
        for st in streams:
            e = torch.cuda.Event()
            e.record(st)
            main.wait_event(e)

    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(9)

    def step_e2e():
        # the three stage families are independent per frame; a replay driver calls the (blocking, host-pointer) ABI
        # entry points from three host threads, one per context / stream (ctypes releases the GIL during the call)
        def e_orb():
            torch.cuda.set_device(local_rank)
            for s in range(SUBS_PER_STEP):
                c_orb.check(L.pslam_orb_extract_batch(c_orb.h, h_gray[s * SUB_BATCH].data_ptr(), SUB_BATCH, h_kps.ctypes.data, h_desc.ctypes.data,
                                                      cap, h_n.ctypes.data))
                if EXTRAS:      # Frame::ComputeStereoFromRGBD on the key points just returned (host buffers in, host buffers out)
                    c_orb.check(L.pslam_compute_stereo_from_rgbd_batch(c_orb.h, h_kps.ctypes.data, h_kps.ctypes.data, h_n.ctypes.data, cap, h_depth[s * SUB_BATCH].data_ptr(),
                                                                       SUB_BATCH, DEPTH_FACTOR, BF, h_ur.ctypes.data, h_dz.ctypes.data))

        def e_peac():
            torch.cuda.set_device(local_rank)
            for s in range(SUBS_PER_STEP):
                if EXTRAS:      # the whole Frame::ComputePlanes: PEAC + post-processing + surface normals -> mvPlaneCoefficients, mvPlanePoints, vSurfaceNormal
                    c_peac.check(L.pslam_compute_planes_batch(c_peac.h, h_depth[s * SUB_BATCH].data_ptr(), SUB_BATCH, DIST_TH, h_pp_n.ctypes.data, h_pp_src.ctypes.data,
                                                              h_pp_coef.ctypes.data, h_pp_off.ctypes.data, h_pp_pts.ctypes.data, PP_CAP, h_sn8.ctypes.data))
                else:
                    c_peac.check(L.pslam_peac_run_batch(c_peac.h, h_depth[s * SUB_BATCH].data_ptr(), SUB_BATCH, h_labels.ctypes.data,
                                                        h_planes.ctypes.data, h_npl.ctypes.data, None, None))

        def e_pose():
            torch.cuda.set_device(local_rank)
            for s in range(SUBS_PER_STEP):
                opt.PoseOptimizationBatch(probs)
        def e_lsd():
            torch.cuda.set_device(local_rank)
            for q in range(LSD_SUBS):
                o, n = q * LSD_BATCH, min(LSD_BATCH, FRAMES_PER_STEP - q * LSD_BATCH)
                if EXTRAS:      # the whole ExtractLineSegment (with LBD descriptors), then Frame::isLineGood on the key lines just returned
                    c_lsd.check(L.pslam_lines_extract_describe_batch(c_lsd.h, h_gray[o].data_ptr(), n, MAX_LINES, h_kl[o:].ctypes.data, h_lf[o:].ctypes.data,
                                                                     h_ldesc[o:].ctypes.data, None, h_nkl[o:].ctypes.data))
                    c_lsd.check(L.pslam_lines3d_batch(c_lsd.h, h_kl[o:].ctypes.data, h_nkl[o:].ctypes.data, MAX_LINES, h_depth[o].data_ptr(), n, DEPTH_FACTOR, cam4,
                                                      h_seed[o:].ctypes.data, None, h_l3d[o:].ctypes.data, h_drawn[o:].ctypes.data))
                else:
                    c_lsd.check(L.pslam_lines_extract_batch(c_lsd.h, h_gray[o].data_ptr(), n, MAX_LINES, h_kl[o:].ctypes.data, h_lf[o:].ctypes.data,
                                                            h_nkl[o:].ctypes.data))
        fns = [fn for nm, fn in (("peac", e_peac), ("lsd", e_lsd), ("orb", e_orb), ("pose", e_pose)) if nm in STAGES]
        for f in [pool.submit(fn) for fn in fns]:
            f.result()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def dump_last_step():
        """What the last timed step left in the stage buffers: ORB, PEAC and pose hold the step's last sub-batch, LSD every frame of the step.  A fixed
        sample of frames (seed 0) keeps the files small; entries past a frame's count are zeroed, since the buffers are reused without clearing."""
        torch.cuda.synchronize(dev)
        rng = np.random.default_rng(0)
        sb = np.sort(rng.choice(SUB_BATCH, min(8 // AREA, SUB_BATCH), replace=False))            # frames of the last sub-batch (image-sized outputs)
        fs = np.sort(rng.choice(FRAMES_PER_STEP, min(64, FRAMES_PER_STEP), replace=False))        # frames of the step (LSD)
        last = (SUBS_PER_STEP - 1) * SUB_BATCH
        host = lambda t, rows: t[torch.as_tensor(rows, device=dev)].cpu().numpy()

        def upto(a, n):
            a = a.copy()
            for i, k in enumerate(n):
                a[i, int(k):] = 0
            return a
        out = {}
        if "orb" in STAGES:
            n_all = d_n.cpu().numpy()
            n = n_all[last + sb]
            out["orb_n"] = n_all[last:last + SUB_BATCH]
            out["orb_keypoints"] = upto(host(d_kps, sb).view(KEYPOINT_DTYPE)[..., 0], n)
            out["orb_descriptors"] = upto(host(d_desc, sb), n)
            if EXTRAS:
                out["stereo_u_right"], out["stereo_depth"] = upto(host(d_ur, sb), n), upto(host(d_dz, sb), n)
                q = sb[sb < SUB_BATCH - 1]                                   # MatchORBPoints: frame q + 1 against frame q
                out["match_knn_idx"] = upto(host(d_midx, q), n_all[last + q + 1])
                out["match_knn_dist"] = upto(host(d_mdist, q), n_all[last + q + 1])
                ngood = d_ngood.cpu().numpy()[:SUB_BATCH - 1]
                out["match_n_good"] = ngood
                out["match_good"] = upto(host(d_good, q), ngood[q])               # the gated MatchORBPoints result
                if xch is not None:                                               # key-frame exchange of the step's first sub-batch, every key frame
                    kf = np.minimum(np.arange(KF) * kf_stride, SUB_BATCH - 1)
                    out["exchange_idx"] = upto(d_xidx.cpu().numpy(), n_all[kf])
                    out["exchange_dist"] = upto(d_xdist.cpu().numpy(), n_all[kf])
        if "peac" in STAGES:
            npl_all = d_npl.cpu().numpy()
            npl = npl_all[last + sb]
            moff = upto(host(d_moff, sb), npl + 1)
            out["peac_n_planes"] = npl_all[last:last + SUB_BATCH]
            out["peac_planes"] = upto(host(d_planes, sb).view(PLANE_DTYPE)[..., 0], npl)
            out["peac_labels"] = host(d_labels, sb)
            out["peac_member_offsets"] = moff
            out["peac_members"] = upto(host(d_members, sb), moff[np.arange(len(sb)), npl])
            if EXTRAS:
                pn = host(d_pp_n, sb)
                poff = upto(host(d_pp_off, sb), pn + 1)
                out["planes_n"], out["planes_src"], out["planes_coef"] = pn, upto(host(d_pp_src, sb), pn), upto(host(d_pp_coef, sb), pn)
                out["planes_point_offsets"], out["planes_points"] = poff, upto(host(d_pp_pts, sb), poff[np.arange(len(sb)), pn])
                out["planes_status"] = d_pp_status.cpu().numpy()
                out["surface_normals"] = host(d_sn3, sb)
                out["surface_normal_records"] = host(d_sn8, sb)                   # normal, cameraPosition, FramePosition
                out["manhattan"] = host(d_mres, sb).view(MANHATTAN_RESULT_DTYPE)[..., 0]
                out["manhattan_normal_mask"], out["manhattan_direction_mask"] = host(d_nmask, sb), host(d_dmask, sb)
        if "lsd" in STAGES:
            nkl = d_nkl.cpu().numpy()[fs]
            out["lsd_n_lines"] = d_nkl.cpu().numpy()
            out["lsd_keylines"] = upto(host(d_kl, fs).view(KEYLINE_DTYPE)[..., 0], nkl)
            out["lsd_line_functions"] = upto(host(d_lf, fs), nkl)
            if EXTRAS:
                out["lsd_descriptors"] = upto(host(d_ldesc, fs), nkl)
                l3 = upto(host(d_l3d, fs).view(LINE3D_DTYPE)[..., 0], nkl)
                out["lines3d"] = l3[[f for f in LINE3D_DTYPE.names if f != "inliers"]]
                out["lines3d_inliers_u32"] = np.ascontiguousarray(l3["inliers"]).view(np.uint32).reshape(l3.shape + (2,))       # a 64-bit mask: two exact halves
                out["lines3d_draws"] = d_drawn.cpu().numpy()
        if "pose" in STAGES:
            res = opt.fetch()
            out["pose_Tcw"] = np.stack([r["Tcw_d"] for r in res])
            out["pose_Tcw_float"] = np.stack([r["Tcw"] for r in res])
            out["pose_n_inliers"] = np.array([r["n_inliers"] for r in res], np.int32)
            out["pose_trace_i"], out["pose_trace_d"] = np.stack([r["trace_i"] for r in res]), np.stack([r["trace_d"] for r in res])
            for k in ("outlier_pt", "outlier_line", "outlier_plane", "outlier_par", "outlier_ver"):
                out["pose_" + k] = np.concatenate([res[i][k] for i in sb])
        total = save_outputs(args.dump_outputs, out)
        print(f"bench: {len(out)} outputs of the last timed step ({total} bytes) written to {args.dump_outputs}", file=sys.stderr)

    # ---- device-resident throughput ----
    steps_dev(max(args.warmup, 3))
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = sum(c.launch_count for c in ctxs)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(main)
    steps_dev(args.steps)
    e1.record(main)
    barrier()
    sampler.stop_flag = True
    launches = sum(c.launch_count for c in ctxs) - l0
    ms = e0.elapsed_time(e1)
    n_found = int(d_n.sum().item())
    n_planes_found = int(d_npl.sum().item())
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * FRAMES_PER_STEP * args.steps / (ms_max / 1e3)
    if args.dump_outputs:
        if rank == 0:
            dump_last_step()
        barrier()                  # the other ranks' next exchange waits on rank 0's epoch flag: keep them from starting it during the dump

    # ---- per-kernel roofline pass (event-bracketed launches, same workload, outside the timed regions) ----
    # one stage family at a time, so a launch's duration is not inflated by kernels of the other two streams
    rep = {}
    for nm, c, fn in (("orb", c_orb, lambda: dev_orb(0)), ("lsd", c_lsd, dev_lsd), ("peac", c_peac, lambda: dev_peac(0)),
                      ("pose", c_pose, opt.run_packed)):
        if nm not in STAGES:
            continue
        c.profile(True)
        for _ in range(1 if nm == "lsd" else SUBS_PER_STEP):       # dev_lsd() without argument runs its LSD_SUBS calls
            fn()
        torch.cuda.synchronize(dev)
        rep.update(c.profile_report())
        c.profile(False)
    peak, peak_kind = _peaks()
    per_kernel = {}
    for name, (n, tot_ms) in rep.items():
        frames_per_launch = FRAMES_PER_STEP / n
        bytes_per_launch = ALGO_BYTES.get(name, 0) * AREA * frames_per_launch
        if name.startswith("exchange_"):           # one key frame per launch (the matcher reads one record per rank)
            bytes_per_launch = ALGO_BYTES[name] * (world if name == "exchange_match" else 1)
        per_kernel[name] = {"launches": n, "ms_total": round(tot_ms, 4), "share": None, "algo_bytes_per_launch": int(bytes_per_launch),
                            "achieved_gbs": round(bytes_per_launch / (tot_ms / n * 1e-3) / 1e9, 2)}
    tot = sum(v["ms_total"] for v in per_kernel.values()) or 1.0
    for v in per_kernel.values():
        v["share"] = round(v["ms_total"] / tot, 4)
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms_total"])
    # DRAM bytes per frame of the dominant kernels from the committed round-2 `ncu --set full` captures (dram__bytes_read.sum + dram__bytes_write.sum of one
    # launch / its frames: profiles/r2_ncu_full_lsd_kernels.csv at 3552 frames, profiles/r2_ncu_full_peac_kernels.csv at 1776; k_peac_flood from
    # profiles/r1_ncu_full_summary.csv at 296 - its round-2 capture returned no DRAM counters), scaled to this run's frames per launch
    # (k_lsd_regions re-captured after its last change at the benchmark launch size: 99.141 + 9.583 GB per 3552 frames, profiles/r2_final_ncu_full_lsd_regions_peac_flood.csv)
    NCU_DRAM_BYTES_PER_FRAME = {"lsd_regions": (99.140878e9 + 9.582504e9) / 3552, "peac_cluster": (8.573231e9 + 3.334866e9) / 1776,
                                "peac_flood": (4.953115e9 + 1.131992e9) / 296, "lsd_improve": (3.480971e9 + 1.401838e9) / 3552}
    traffic = NCU_DRAM_BYTES_PER_FRAME.get(dom)
    roofline = {"kernel": dom, "bound": "hbm", "achieved": per_kernel[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": round(per_kernel[dom]["achieved_gbs"] / peak, 6),
                "traffic": int(traffic * FRAMES_PER_STEP / per_kernel[dom]["launches"]) if traffic else None, "peak_kind": peak_kind,
                "note": "serial-order kernels (quadtree, AHC, PEAC / LSD region growing, LM) run one warp/CTA per frame: latency-bound, see DESIGN.md",
                "per_kernel": per_kernel}

    # ---- auxiliary: LocalBundleAdjustment throughput (BASELINE.json config 4: 20 KFs, 5000 point + 200 line + 30 plane edges) ----
    aux = {}
    try:
        from planarslam_b200 import synth_lba
        from planarslam_b200.lba import LocalBundleAdjuster
        n_lba = 296
        base = [synth_lba.make_lba_problem(k) for k in range(4)]
        ba = LocalBundleAdjuster(c_pose)
        ba.pack([base[k % 4] for k in range(n_lba)])
        ba.run_packed()
        torch.cuda.synchronize(dev)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(streams[2]):
            a0.record()
            for _ in range(3):
                ba.run_packed()
            a1.record()
        torch.cuda.synchronize(dev)
        aux["local_bundle_adjustments_per_sec"] = round(3 * n_lba / (a0.elapsed_time(a1) * 1e-3), 1)
        aux["lba_config"] = "20 key frames (1 fixed), 5000 point + 100 line (200 edges) + 30 plane-type edges, 296 problems per launch"
    except Exception as ex:                      # auxiliary only: never fail the headline
        aux["lba_error"] = repr(ex)
    # ---- auxiliary: Frame::isLineGood and Tracking::TrackManhattanFrame (kernels added after the round-1 GPU budget was spent): run in a
    # child process so that a fault there cannot touch this process' CUDA context; it reports throughput and whether the results match
    # the signatures computed on the CPU at commit time (tests/golden/aux_new_kernels_expected.json) ----
    if rank == 0 and os.environ.get("PSLAM_AUX_NEW", "1") != "0":
        import subprocess
        try:
            env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "aux_new_kernels.py")], capture_output=True, text=True, timeout=150, env=env)
            if r.returncode == 0 and r.stdout.strip():
                aux["new_kernels"] = json.loads(r.stdout.strip().splitlines()[-1])
            else:
                aux["new_kernels"] = {"error": f"exit code {r.returncode}", "stderr": r.stderr[-300:]}
        except Exception as ex:
            aux["new_kernels"] = {"error": repr(ex)}

    xch_info = None
    if xch is not None:
        n_to = C.c_int32(0)
        L.pslam_exchange_timeouts.argtypes = [C.c_void_p, C.c_void_p]
        c_orb.check(L.pslam_exchange_timeouts(c_orb.h, C.byref(n_to)))
        if n_to.value:
            raise RuntimeError(f"key-frame exchange: {n_to.value} matcher CTAs timed out waiting for a peer")
        xch_info = {"key_frames_per_rank_per_step": KF, "records_read_per_match": world, "transport": "CUDA IPC peer memory (NVLink P2P), fused with the Hamming k=2 matcher",
                    "epochs": xch_epoch[0], "second_nearest_distance_median": float(d_xdist[:, :500, 1].float().median().item())}
    # ---- end to end through the host-pointer ABI ----
    n_keylines = float(d_nkl.sum().item()) if "lsd" in STAGES else None
    frame_e2e = EXTRAS and all(k in STAGES for k in ("orb", "lsd", "peac"))
    if frame_e2e:
        # The call a replay driver makes per batch is the Frame constructor's compute, pslam_frame_construct_batch: host frames in (uploaded once), every Frame
        # product out.  Two contexts on two host threads take alternate sub-batches, so one batch's copies overlap the other's kernels; PoseOptimization runs on
        # a third thread as before.  The device-resident leg's contexts and buffers are released first (two full-family contexts take ~110 GB).
        barrier()
        xch = None
        del d_gray, d_depth, d_kps, d_desc, d_labels, d_planes, d_members, d_moff, d_kl, d_lf, d_ur, d_dz, d_midx, d_mdist, d_good, d_ldesc, d_l3d, d_pp_coef, d_pp_pts
        del d_sn8, d_sn3, d_nmask
        for c in (c_orb, c_peac, c_lsd):
            c.close()
        torch.cuda.empty_cache()
        from planarslam_b200.frame import ConstructFrames, FrameOutputs
        # PSLAM_E2E_CONTEXTS contexts (default 2) of 2 * SUB_BATCH / contexts frames each - the device memory of two full sub-batches either way.  Measured on B200
        # (profiles/r2_exp_e2e_*contexts.json): two contexts of 1776 frames 5.2 k frames/s, four of 888 frames 4.6 k - smaller calls leave the one-warp-per-frame
        # kernels with quarter-wave launches.
        E2E_CTX = max(2, int(os.environ.get("PSLAM_E2E_CONTEXTS", "2")))
        E2E_BATCH = max(1, 2 * min(SUB_BATCH, int(os.environ.get("PSLAM_E2E_WAVE", str(DEFAULT_WAVE)))) // E2E_CTX)      # (two contexts of one clustering wave each: ~110 GB)
        E2E_CALLS = (FRAMES_PER_STEP + E2E_BATCH - 1) // E2E_BATCH
        fctx = [Context(W, H, E2E_BATCH, device=local_rank, nfeatures=NFEATURES) for _ in range(E2E_CTX)]
        fout = [FrameOutputs(c, E2E_BATCH, MAX_LINES, PP_CAP, normals=True, pinned=True) for c in fctx]

        def e_frames(t):
            torch.cuda.set_device(local_rank)
            for sb in range(t, E2E_CALLS, E2E_CTX):
                o = sb * E2E_BATCH
                ConstructFrames(fctx[t], h_gray[o].data_ptr(), h_depth[o].data_ptr(), fout[t], DEPTH_FACTOR, BF, DIST_TH, 1, nframes=min(E2E_BATCH, FRAMES_PER_STEP - o))

        # PoseOptimization through the host-pointer batch call of the C ABI: the problem descriptors (plain structs pointing at the host arrays) are built once -
        # the call itself packs the edge records from the host arrays, uploads them, optimises and returns poses / outlier flags / inlier counts every time
        from planarslam_b200.optimizer import _to_struct
        from planarslam_b200._lib import PoseProblem
        pose_arr = (PoseProblem * len(probs))(*[_to_struct(p_) for p_ in probs])
        pose_T0 = np.ascontiguousarray(np.stack([p_["Tcw0"] for p_ in probs]), np.float32)
        pose_T = np.empty_like(pose_T0)
        pose_flags = [np.zeros(max(sum(len(p_[k]) for p_ in probs), 1), np.uint8) for k in ("Xw", "line_Xw", "plane_meas", "par_meas", "ver_meas")]
        pose_ninl = np.zeros(len(probs), np.int32)
        L.pslam_pose_optimization_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 7

        def e_pose2():
            torch.cuda.set_device(local_rank)
            for _ in range(SUBS_PER_STEP):
                np.copyto(pose_T, pose_T0)
                c_pose.check(L.pslam_pose_optimization_batch(c_pose.h, pose_arr, len(probs), pose_T.ctypes.data, *[f_.ctypes.data for f_ in pose_flags], pose_ninl.ctypes.data))

        def step_e2e():
            jobs = [pool.submit(e_frames, t) for t in range(E2E_CTX)] + ([pool.submit(e_pose2)] if "pose" in STAGES else [])
            for f in jobs:
                f.result()
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(2, args.steps // 3)
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = world * FRAMES_PER_STEP * e2e_steps / float(t.item())
    if frame_e2e:
        h2d = FRAMES_PER_STEP * 3 * W * H + ("pose" in STAGES) * SUBS_PER_STEP * pose_h2d
        d2h = E2E_CALLS * fout[0].nbytes() + ("pose" in STAGES) * FRAMES_PER_STEP * (64 + 1046 + 4)
        e2e_call = (f"pslam_frame_construct_batch (Frame constructor: one upload of gray + depth per frame) on {E2E_CTX} contexts / host threads, {E2E_BATCH} frames per call "
                    "+ pslam_pose_optimization_batch")
    else:
        h2d = FRAMES_PER_STEP * (("orb" in STAGES) * W * H + ("lsd" in STAGES) * W * H + ("peac" in STAGES) * 2 * W * H) + ("pose" in STAGES) * SUBS_PER_STEP * pose_h2d
        d2h = FRAMES_PER_STEP * (("orb" in STAGES) * (cap * 60 + 8) + ("peac" in STAGES) * (4 * W * H + maxp * PLANE_DTYPE.itemsize + 4) +
                                 ("pose" in STAGES) * (64 + 1046 + 4) + ("lsd" in STAGES) * (MAX_LINES * (68 + 24) + 4))
        if EXTRAS:          # stereo: key points + depth again; isLineGood: key lines + depth again (every host-pointer call uploads what it reads)
            h2d += FRAMES_PER_STEP * (("orb" in STAGES) * (cap * 28 + 2 * W * H) + ("lsd" in STAGES) * (MAX_LINES * 68 + 2 * W * H))
            d2h += FRAMES_PER_STEP * (("orb" in STAGES) * cap * 8 + ("lsd" in STAGES) * MAX_LINES * (32 + 96) +
                                      ("peac" in STAGES) * (maxp * 28 + 4096 * 12 + n_sn * 32 - 4 * W * H - maxp * PLANE_DTYPE.itemsize))
        e2e_call = "per-function host-pointer entry points, one host thread per stage family"

    if frame_e2e:            # the end-to-end contexts are no longer needed: the tracking-chain measurement below runs on an otherwise idle GPU
        for c in fctx:
            c.close()
        torch.cuda.empty_cache()
    # ---- auxiliary: BASELINE.json config 3, the device-resident tracking chain on ONE sequence (frame t+1 needs the pose of frame t: a latency number) ----
    if rank == 0:
        try:
            from planarslam_b200 import synth, synth_map
            from planarslam_b200.orb import ORBextractor
            from planarslam_b200.tracking import Tracker
            nseq = 64
            fr = [synth.render_frame(2, f)[:2] for f in range(nseq)]
            ex = ORBextractor(1000, 1.2, 8, 20, 7)
            parts = []
            for f in range(0, nseq, 8):
                k, de = ex(fr[f][0])
                parts.append(synth_map.map_from_frame(synth_map.frame_arrays(k, de, fr[f][1]), synth_map.true_pose(f)))
            m = {key: np.concatenate([q[key] for q in parts]) for key in ("pos", "normal", "max_distance", "min_distance", "desc", "skip", "has_obs")}
            tctx = Context(640, 480, max_batch=nseq, device=local_rank)
            tr = Tracker(tctx)
            tr.set_map(m)
            sg, sd, T0 = np.stack([f[0] for f in fr]), np.stack([f[1] for f in fr]), synth_map.true_pose(0).astype(np.float32)
            tr.track(sg, sd, T0)
            t0 = time.perf_counter()
            poses, stats = tr.track(sg, sd, T0)
            dt = time.perf_counter() - t0
            err = max(synth_pose.pose_error(poses[t], synth_map.true_pose(t))[0] for t in range(nseq))
            aux["tracking_chain"] = {"frames_per_sec_single_sequence": round(nseq / dt, 1), "frames": nseq, "map_points": int(len(m["skip"])),
                                     "max_rotation_error_vs_ground_truth_rad": float(err), "min_inliers": int(stats[:, 3].min()),
                                     "what": "ORB -> stereo -> motion model -> SearchByProjection(last) -> PoseOptimization -> SearchByProjection(map) -> PoseOptimization, host frames in"}
            tctx.close()
        except Exception as ex_:
            aux["tracking_chain"] = {"error": repr(ex_)}
    if rank == 0:
        modes = cpu_modes(gray[:CPU_SAMPLE_FRAMES], depth[:CPU_SAMPLE_FRAMES], seconds=float(os.environ.get("PSLAM_CPU_SECONDS", "8")))
        best = modes["frame_parallel_all_cores"]
        line = {"metric": f"rgbd_frames_per_sec_{W}x{H}", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic", "config": workload_config(),
                "clocks": sampler.summary(), "gpu_launches": int(launches),
                "e2e": {"value": e2e_val, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "call": e2e_call},
                "roofline": roofline,
                "cpu_baseline": {"value": best["frames_per_sec"], "unit": "frames/s", "cores": best["threads"], "kind": "reference",
                                 "units": {k: CPU_UNITS.get(k) for k in STAGES}, "modes": modes,
                                 "sample": f"{' + '.join(STAGES)}: {best['frames']} frames in {best['seconds']} s, one pinned process per host core "
                                           f"({modes['host_cores']}), -O3 -march=x86-64-v3 (oracle/Makefile fast); modes = BASELINE.md section 3"},
                "keypoints_per_frame": n_found / FRAMES_PER_STEP, "planes_per_frame": n_planes_found / FRAMES_PER_STEP,
                "keylines_per_frame": n_keylines / FRAMES_PER_STEP if n_keylines is not None else None, "exchange": xch_info, "aux": aux}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
