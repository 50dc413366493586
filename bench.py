#!/usr/bin/env python3
"""bench.py -- headline benchmark of the ygz-slam hot path on B200 (contract: task statement, section 4).

Workload (BASELINE.json metric "tracked frames/sec on 640x480 synthetic stream", configs[4] "C5"): `--streams` (8)
independent synthetic 640x480 streams per GPU through the FULL tracking loop of the reference --
    Frame::InitFrame (pyramid) -> Matcher::SparseImageAlignment against the reference key-frame
    -> LocalMapping::TrackLocalMap: candidate projection + Matcher::FindDirectProjection (8x8 patch alignment) of the
       local map -> ba::OptimizeCurrentPoseOnly -> key-frame decision
    -> at key-frames FeatureDetector::Detect (grid FAST-10 + ORB), depth-initialised map points, ba::LocalBAG2O.
One STEP = `--frames-per-step` (10) consecutive frames of every stream (80 tracked frames per GPU); every step consumes
frames that were never touched before.  metric = tracked frames/sec (whole job, all ranks).

  value : frames already resident in HBM when the timed region starts; the region is timed with CUDA events on the
          library's stream (first event after the warm-up barrier, second after every stream has drained), max over ranks.
  e2e   : the same loop through the public C ABI with HOST buffers: every step's frames are copied from pinned host
          memory (H2D) and the poses / features / BA results are read back (D2H) inside the timed region.
  roofline      : dominant kernel of the step (largest share of the device time, CUDA events around each launch in a
                  separate profiled pass) -- algorithmic bytes / duration against MEASURED_PEAKS.json hbm_gbs, plus the
                  FP64 FLOP/s of the BA reduce.
  cpu_baseline  : the CPU oracle (-O3 AVX2/FMA build of the reference restatement) through the same loop in C++
                  (oracle/vo_cpu.cpp) on a bounded sample of the same streams, rank 0, N=1 only; 1 thread and
                  one thread per stream, with a per-stage breakdown.
  --impl reference : the reference's CPU path (oracle restatement: the reference itself cannot be built here) through
                  the same loop on all usable host threads, one independent stream per thread, same metric/config.
  --workload extract_match : BASELINE configs[1] (C2, the round-1 headline); at N=1 it is also run as a secondary record.
Multi-GPU: independent streams per rank, no data-path collective ("weak" scaling: 8 streams per GPU); the BASELINE
sentence "8 streams sharded across the GPUs" is measured as well (`sharded_8_streams`, 8/N streams per GPU).
torch.distributed (NCCL) only for the barrier, the max-over-ranks of the device time and the gather of per-rank records.
"""
from __future__ import annotations

import os as _os

# Every engine thread owns two CUDA streams (tracking chain + upload / alignment); with the default 8 hardware work queues
# ("connections") the streams of several threads share a queue and falsely serialise behind each other -- measured: 8 host
# threads 22k tracked frames/s with 8 connections, 28.6k with 32, and the rare 5x slow legs disappear.  Must be set before the
# CUDA context exists, i.e. before torch / the library touch the device.
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

W, H, LEVELS = 640, 480, 8
FRAME_BYTES = W * H
PYR_BYTES = sum(((W + (1 << L) - 1) >> L) * ((H + (1 << L) - 1) >> L) for L in range(LEVELS))  # 409,600


def make_frames(n: int, seed: int) -> np.ndarray:
    """n distinct 640x480 grey frames: sliding crops of one perspective render + per-frame noise."""
    from ygz_slam_b200 import synth
    tex = synth.texture(0x59475A00 + seed, 2048)
    bw, bh = W + 512 + 16, H + 64          # 1168 x 544 px at z = 2 m stays inside the 5.12 m texture
    base, _ = synth.render_plane(tex, synth.trajectory(seed), w=bw, h=bh, cx=bw / 2, cy=bh / 2)
    rng = np.random.default_rng(seed + 1)
    out = np.empty((n, H, W), np.uint8)
    for k in range(n):
        x0, y0 = (2 * k) % 512, (7 * k) % 64
        crop = base[y0:y0 + H, x0:x0 + W].astype(np.int16)
        crop += np.rint(rng.normal(0, 2.0, (H, W))).astype(np.int16)
        out[k] = np.clip(crop, 0, 255).astype(np.uint8)
    return out


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML; same fields as the profiling
    guide's nvidia-smi line: clocks.sm, clocks.max.sm, clocks_event_reasons.*)."""

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = self.gpu_index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu_index])
                except (ValueError, IndexError):
                    pass
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.err = f"nvml unavailable: {e}"
            return
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                "hw_power_brake": 0x80}

        def loop():
            while not self._stop.is_set():
                try:
                    self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    try:
                        r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:  # noqa: BLE001
                        r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for name, bit in bits.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception as e:  # noqa: BLE001
                    self.err = str(e)
                    return
                time.sleep(0.02)

        self._thr = threading.Thread(target=loop, daemon=True)
        self._thr.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=1.0)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "samples": 0, "reasons": [self.err or "no samples"]}
        s = sorted(self.samples)
        load = s[len(s) // 2:]  # the busier half of the samples = under load
        return {"sm_mhz": float(np.median(load)), "sm_mhz_min": s[0], "sm_max_mhz": self.max_mhz, "samples": len(s),
                "reasons": sorted(self.reasons)}


def bind_to_gpu_numa(gpu_index: int) -> dict:
    """Pin this process (and the host threads it creates later: the C++ drivers' workers inherit the mask) to the CPUs that are
    local to its GPU's PCIe root, so that pinned frame buffers are allocated on, and copied from, the GPU's own NUMA node.
    8 ranks on one box otherwise share whatever node the scheduler picks (round 1: e2e scaling 0.59 at N=8)."""
    info = {"bound": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        idx = gpu_index
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                idx = int(vis.split(",")[gpu_index])
            except (ValueError, IndexError):
                pass
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
        if isinstance(bus, bytes):
            bus = bus.decode()
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{int(dom, 16):04x}:{rest.lower()}"
        cpus = set()
        for part in open(path + "/local_cpulist").read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        info["numa_node"] = int(open(path + "/numa_node").read().strip())
        allowed = os.sched_getaffinity(0) & cpus
        info["local_cpus"] = len(cpus)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["bound"] = True
            info["cpus_bound"] = len(allowed)
    except Exception as e:  # noqa: BLE001 -- binding is an optimisation, never a failure
        info["error"] = repr(e)
    return info


def measured_peaks() -> tuple:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------
def cpu_run(ora, frames: np.ndarray, count: int, threads: int):
    """Reference CPU path (pyramid + Detect + cross-checked BF match of frame k against k+1) for `count` frames on
    `threads` C++ threads (oracle/bench_driver.cpp; no Python inside the timed region).  Returns (seconds, features)."""
    import ctypes as C
    fn = ora.lib.ora_bench_extract_match
    fn.restype = C.c_double
    nf = C.c_long(0)
    frames = np.ascontiguousarray(frames)
    dt = fn(frames.ctypes.data_as(C.c_void_p), len(frames), W, H, LEVELS, int(count), int(threads), C.byref(nf))
    return dt, nf.value


def run_reference(args, rank: int, world: int) -> None:
    """--impl reference: CPU path on all host threads (rank 0 only prints)."""
    if rank != 0:
        return
    from oracle.pyoracle import Oracle
    ora = Oracle(native=True)
    # all the host threads the process may use: the scheduler affinity mask, capped by a cgroup CPU quota if there is one
    threads, usable, quota = usable_threads()
    n = 512                             # the same 512-frame batch per step as the GPU arm (frame-parallel over the threads)
    per_thread = -(-n // threads)
    frames = make_frames(n, 0)
    for _ in range(args.warmup):
        cpu_run(ora, frames, n, threads)
    dt = 0.0
    for _ in range(args.steps):
        dt += cpu_run(ora, frames, n, threads)[0]
    fps = n * args.steps / dt
    line = {
        "impl": "reference", "metric": "tracked frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(n, "C++ host threads, frame-parallel (oracle/bench_driver.cpp)"),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": f"{n} frames/step (<= {per_thread} per thread) x {args.steps} steps; CPU restatement of the reference "
                                   f"path (the reference cannot be built here), -O3 AVX2/FMA, {threads} std::threads",
                         "logical_cpus": os.cpu_count(), "affinity_cpus": usable, "cgroup_cpu_quota": quota},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def secondary_workloads(ctx) -> dict:
    """BASELINE configs C3 (alignment) and C4 (local BA) on one GPU next to the CPU oracle (rank 0, N=1 only).
    Timed through the public C ABI (host buffers in, host buffers out), CUDA kernels timed by the library's
    per-stage events."""
    import numpy as np
    from oracle.pyoracle import Oracle
    from ygz_slam_b200 import se3, synth
    ora = Oracle(native=True)
    out = {}
    # ---- C3: 2000 8x8 patches (FindDirectProjection) + sparse image alignment, 4-level pyramid --------
    g1, d1, T1 = synth.stream_frame(1)
    g2, _, T2 = synth.stream_frame(4)
    fr = ctx.frames(2)
    fr.upload(np.stack([g1, g2]))
    p1, p2 = ora.build_pyramid(g1, LEVELS), ora.build_pyramid(g2, LEVELS)
    f = ora.detect(p1, n_levels=LEVELS)
    rng = np.random.default_rng(7)
    idx = rng.integers(0, f["n"], 2000)
    px = np.stack([f["px"][idx], f["py"][idx]], 1)
    depth = d1[px[:, 1].astype(int), px[:, 0].astype(int)]
    level = f["level"][idx]
    Trel = se3.mul(T2, se3.inv(T1))
    Xc = np.stack([(px[:, 0] - synth.CX) * depth / synth.FX, (px[:, 1] - synth.CY) * depth / synth.FY, depth], 1)
    Xc2 = (Trel[:, :3] @ Xc.T).T + Trel[:, 3]
    gt = np.stack([synth.FX * Xc2[:, 0] / Xc2[:, 2] + synth.CX, synth.FY * Xc2[:, 1] / Xc2[:, 2] + synth.CY], 1)
    init = gt + rng.uniform(-2, 2, gt.shape)
    I = np.eye(4)[:3]
    poses = np.stack([I.reshape(-1), Trel.reshape(-1)])
    z, o = np.zeros(2000, np.int32), np.ones(2000, np.int32)

    def timed(fn, reps):
        fn()
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        return (time.perf_counter() - t0) / reps, r

    ctx.profile(True)
    t_gpu, (gpx, glvl, gok) = timed(lambda: fr.project_align(z, o, poses, z, o, px, depth, level.astype(np.uint8), init), 20)
    prof = ctx.profile_read()
    t_cpu, (cpx, clvl, cok) = timed(lambda: ora.find_direct_projection(p1, p2, W, H, LEVELS, I, Trel, px, depth, level, init), 3)
    spx, slvl, sok = Oracle(native=False).find_direct_projection(p1, p2, W, H, LEVELS, I, Trel, px, depth, level, init)
    out["c3_project_align_2000_patches"] = {
        "gpu_ms_per_call_e2e": t_gpu * 1e3, "gpu_kernel_ms": prof["project_align"][0] / max(prof["project_align"][1], 1),
        "cpu_ms_per_call": t_cpu * 1e3, "patches_per_s_gpu_e2e": 2000 / t_gpu,
        # parity is defined against the unfused (-ffp-contract=off) oracle build; the timed CPU leg is the -O3/FMA build
        "bit_exact_vs_oracle": bool(np.array_equal(gpx, spx) and np.array_equal(gok, sok) and np.array_equal(glvl, slvl)),
        "max_px_diff_vs_fma_build": float(np.max(np.abs(gpx - cpx)[gok & cok])) if (gok & cok).any() else None,
        "converged": int(gok.sum())}
    has = np.ones(2000, np.uint8)
    t_gpu, (gT, gn, _) = timed(lambda: fr.sparse_align([0], [1], [0, 2000], px, depth, has, T1.reshape(1, 12), T1.reshape(1, 12), max_level=3), 20)
    prof = ctx.profile_read()
    t_cpu, (cT, cn, _) = timed(lambda: ora.sparse_align(p1, p2, W, H, LEVELS, px, depth, has, T1, T1, max_level=3), 3)
    out["c3_sparse_align_2000_features_4_levels"] = {
        "gpu_ms_per_call_e2e": t_gpu * 1e3, "gpu_kernel_ms": prof["sparse_align"][0] / max(prof["sparse_align"][1], 1),
        "cpu_ms_per_call": t_cpu * 1e3,
        "pose_diff_vs_oracle": float(np.linalg.norm(se3.se3_log(se3.mul(se3.inv(gT[0]), cT)))),
        "pose_err_vs_ground_truth": float(np.linalg.norm(se3.se3_log(se3.mul(se3.inv(gT[0]), T2))))}
    fr.close()
    # ---- C4: local BA 10 KF x 2000 landmarks x ~8000 observations, 20 LM iterations, Huber 5.991 -------
    sc = synth.ba_scene()
    g2o = np.concatenate([sc["poses_noisy"][:, 3:], sc["poses_noisy"][:, :3]], 1)
    fixed = np.zeros(10, np.uint8)
    fixed[0] = 1
    n_obs = len(sc["kf_idx"])
    t_gpu, (P, X, outl, st) = timed(lambda: ctx.local_ba([0, 10], [0, 2000], [0, n_obs], g2o, fixed, sc["pts_noisy"], sc["kf_idx"],
                                                         sc["pt_idx"], sc["px"]), 10)
    prof = ctx.profile_read()
    ctx.profile(False)
    t_cpu, (wP, wX, wout, wst) = timed(lambda: ora.local_ba(g2o, fixed, sc["pts_noisy"], sc["kf_idx"], sc["pt_idx"], sc["px"]), 3)
    k_ms = prof["local_ba"][0] / max(prof["local_ba"][1], 1)
    # the Ceres flavour (ba::LocalBA, "vs CPU Ceres" of BASELINE.json): same scene, poses as [t; angle-axis]
    t_aa = []
    for v in sc["poses_noisy"]:
        Tm = se3.se3_exp(v)
        t_aa.append(np.r_[Tm[:, 3], se3.so3_log(Tm[:, :3])])
    t_aa = np.array(t_aa)
    ctx.profile(True)
    t_gpu_c, (cP, cX, cst) = timed(lambda: ctx.local_ba_ceres([0, 10], [0, 2000], [0, n_obs], t_aa, fixed, sc["pts_noisy"], sc["kf_idx"],
                                                              sc["pt_idx"], sc["px"]), 10)
    prof_c = ctx.profile_read()
    ctx.profile(False)
    t_cpu_c, (wcP, wcX, wcst) = timed(lambda: ora.local_ba_ceres(t_aa, fixed, sc["pts_noisy"], sc["kf_idx"], sc["pt_idx"], sc["px"]), 3)
    kc_ms = prof_c["local_ba"][0] / max(prof_c["local_ba"][1], 1)
    out["c4_local_ba_ceres_twin"] = {
        "gpu_ms_total_e2e": t_gpu_c * 1e3, "gpu_kernel_ms_total": kc_ms, "gpu_iters": cst[0]["iters"],
        "gpu_ms_per_iter": kc_ms / max(cst[0]["iters"], 1), "cpu_ms_total": t_cpu_c * 1e3, "cpu_iters": wcst["iters"],
        "cpu_ms_per_iter": t_cpu_c * 1e3 / max(wcst["iters"], 1),
        "cpu_kind": "oracle restatement of Ceres trust-region LM (forward jets, Schur + dense Cholesky), 1 thread; Ceres itself is not installable here",
        "cost_final_gpu": cst[0]["cost_final"], "cost_final_cpu": wcst["cost_final"], "termination": cst[0]["termination"],
        "max_pose_diff_vs_oracle": float(np.abs(cP - wcP).max()), "max_landmark_diff_vs_oracle_m": float(np.abs(cX - wcX).max())}
    trials = st[0]["lm_trials"]
    kbar = n_obs / 2000.0
    flop_per_trial = 300.0 * n_obs + 2000 * (216 * kbar**2 + 108 * kbar + 50) + 54**3 / 3.0   # SURVEY.md 8d
    out["c4_local_ba_10kf_2000pt"] = {
        "observations": n_obs, "gpu_ms_total_e2e": t_gpu * 1e3, "gpu_kernel_ms_total": k_ms, "gpu_iters": st[0]["iters"],
        "gpu_lm_trials": trials, "gpu_ms_per_iter": k_ms / max(st[0]["iters"], 1), "gpu_ms_per_lm_trial": k_ms / max(trials, 1),
        "cpu_ms_total": t_cpu * 1e3, "cpu_iters": wst["iters"], "cpu_lm_trials": wst["lm_trials"],
        "cpu_ms_per_iter": t_cpu * 1e3 / max(wst["iters"], 1), "cpu_ms_per_lm_trial": t_cpu * 1e3 / max(wst["lm_trials"], 1),
        "cpu_kind": "oracle restatement of g2o LM + Schur (dense Cholesky), 1 thread; Ceres/g2o are not installable here",
        "achieved_gflops_fp64": flop_per_trial * trials / (k_ms * 1e-3) / 1e9, "flop_per_lm_trial_model": flop_per_trial,
        "chi2_final_gpu": st[0]["chi2_final"], "chi2_final_cpu": wst["chi2_final"],
        "max_landmark_diff_vs_oracle_m": float(np.abs(X - wX).max())}
    return out


def opencv_owned_stages(ora) -> dict:
    """The stages the reference delegates to OpenCV (SURVEY 8a: cv::pyrDown Frame.cpp:127-141, cv::BFMatcher
    test_orb_match.cpp:109-131, cv::calcOpticalFlowPyrLK Tracker.cpp:86-133), timed with cv2 itself beside the oracle's port
    of the same arithmetic, on 1 thread and on cv2's default thread count.  cv2 is a timing witness only."""
    try:
        import cv2
    except Exception as e:  # noqa: BLE001
        return {"unavailable": repr(e)}
    from ygz_slam_b200 import synth
    g1, _, _ = synth.stream_frame(1)
    g2, _, _ = synth.stream_frame(3)

    def best(fn, reps=5):
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return 1e3 * min(ts)

    p1, p2 = ora.build_pyramid(g1, LEVELS), ora.build_pyramid(g2, LEVELS)
    f1, f2 = ora.detect(p1, n_levels=LEVELS), ora.detect(p2, n_levels=LEVELS)
    d1 = ora.describe(p1, W, H, LEVELS, f1["px"], f1["py"], f1["level"])[1]
    d2 = ora.describe(p2, W, H, LEVELS, f2["px"], f2["py"], f2["level"])[1]
    n_klt = min(1000, f1["n"])
    pts = np.stack([f1["px"][:n_klt], f1["py"][:n_klt]], 1).astype(np.float32)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING, True)

    def cv_pyr3():
        a = cv2.pyrDown(g1)
        return cv2.pyrDown(a)

    def cv_klt():
        return cv2.calcOpticalFlowPyrLK(g1, g2, pts.reshape(-1, 1, 2), pts.reshape(-1, 1, 2).copy(), winSize=(21, 21), maxLevel=4,
                                        criteria=(cv2.TERM_CRITERIA_COUNT | cv2.TERM_CRITERIA_EPS, 30, 0.001),
                                        flags=cv2.OPTFLOW_USE_INITIAL_FLOW, minEigThreshold=1e-4)

    out = {"inputs": {"image": "640x480 u8", "descriptors": [int(len(d1)), int(len(d2))], "klt_points": int(n_klt)}}
    default_threads = cv2.getNumThreads()
    for label, nt in (("cv2_1_thread_ms", 1), ("cv2_default_threads_ms", default_threads)):
        cv2.setNumThreads(nt)
        out[label] = {"threads": nt, "pyrDown_3_levels": best(cv_pyr3), "BFMatcher_hamming_crosscheck": best(lambda: bf.match(d1, d2)),
                      "calcOpticalFlowPyrLK_21x21_5_levels": best(cv_klt)}
    cv2.setNumThreads(default_threads)
    out["port_1_thread_ms"] = {"threads": 1, "pyrDown_3_levels": best(lambda: ora.build_pyramid(g1, 3)),
                               "BFMatcher_hamming_crosscheck": best(lambda: ora.match_bf(d1, d2)),
                               "calcOpticalFlowPyrLK_21x21_5_levels": best(lambda: ora.klt(g1, g2, pts, pts.copy()), reps=2)}
    out["note"] = ("in the C5 loop only the pyramid is OpenCV-owned (its share is cpu_baseline.stage_share_1_thread.pyramid); the "
                   "matcher and the KLT belong to BASELINE configs C2 and C1")
    return out


def workload_config(batch: int, how: str) -> dict:
    return {"workload": "C2: FAST-10+ORB extract (grid 10px, thr 15) + cross-checked brute-force Hamming match, "
                        "640x480 u8, 8-level pyramid, frame i matched against frame i+1",
            "frames_per_step": batch, "keypoints_per_frame": "~1100-1300 (grid yield on the synthetic stream)",
            "batching": how,
            "l2_policy": "inputs larger than L2: %.0f MB of level-0 pixels per step vs 126 MB L2" % (batch * FRAME_BYTES / 1e6)}



KF_POLICY = dict(kf_min_frames=5, kf_min_rot=0.03, kf_min_trans=0.03)   # as in tests/test_vo.py: a key-frame every >= 5 frames


def usable_threads():
    """Host threads this process may really use: the affinity mask capped by a cgroup CPU quota if there is one."""
    usable = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(p)
    except Exception:  # noqa: BLE001
        pass
    capped = usable if quota is None else max(1, min(usable, int(np.ceil(quota))))
    return capped, usable, quota


def vo_config(streams: int, frames_per_step: int) -> dict:
    """Identical for the GPU arm and the reference arm (the driver compares the two dicts)."""
    return {"workload": "C5: full VO tracking loop on independent synthetic 640x480 u8 streams, 3-level pyramid (reference default): "
                        "sparse image alignment -> direct projection of the local map (8x8 patch alignment) -> pose-only refinement "
                        "-> key-frame decision; key-frames: grid FAST-10 + ORB detect, depth-initialised map points, local BA (g2o "
                        "Levenberg + Schur, 3 local key-frames, 20 iterations)",
            "streams_per_gpu": streams, "frames_per_step_per_stream": frames_per_step,
            "keyframe_policy": "NeedNewKeyFrame: >= %d frames since the last key-frame and rotation > %.2f rad or translation > %.2f m"
                               % (KF_POLICY["kf_min_frames"], KF_POLICY["kf_min_rot"], KF_POLICY["kf_min_trans"]),
            "l2_policy": "every step consumes %d new frames per GPU (%.1f MB of pixels, never re-read); the resident leg keeps all "
                         "(warmup + steps) x that many frames in HBM, larger than the 126 MB L2 for the default steps"
                         % (streams * frames_per_step, streams * frames_per_step * FRAME_BYTES / 1e6)}


def vo_streams(first_stream: int, count: int, n_frames: int):
    from ygz_slam_b200 import synth
    return [synth.shift_stream(first_stream + s, n_frames) for s in range(count)]


def vo_cpu(ora, data, threads: int, warm: int):
    """oracle/vo_cpu.cpp over the given streams; returns (frames/s, seconds, stats, per-stage seconds)."""
    from oracle import pyoracle
    n = len(data[0][0])
    _, stats, sec, stage = pyoracle.vo_run(ora, [d[0] for d in data], [d[1] for d in data], KF_POLICY["kf_min_frames"],
                                           KF_POLICY["kf_min_rot"], KF_POLICY["kf_min_trans"], warm=warm, threads=threads)
    return len(data) * (n - warm) / sec, sec, stats, stage


def run_reference_vo(args, rank: int, world: int) -> None:
    """--impl reference on the VO workload: the C++ loop on the CPU oracle, ONE INDEPENDENT STREAM PER USABLE HOST THREAD (the
    reference tracks one sequence on one thread, so streams are the only parallelism it offers).  The job of the GPU arm has
    8 x n_gpus streams; a host with more threads than that is given more streams (copies of the same pixels, tracked
    independently) so that every thread it can use is busy -- `value` is the box's CPU throughput on this workload.  The
    same-size job (8 x n_gpus streams, one thread each) is reported in cpu_baseline.same_job.  A step = one key-frame cycle
    (5 frames) of every stream: a bounded sample of the GPU arm's 10-frame step."""
    if rank != 0:
        return
    from oracle.pyoracle import Oracle
    ora = Oracle(native=True)
    threads, affinity, quota = usable_threads()
    S, F = args.streams, args.frames_per_step
    Fs = KF_POLICY["kf_min_frames"]                 # frames per stream of one reference-arm step
    n = (args.warmup + args.steps) * Fs
    warm = args.warmup * Fs
    job_streams = S * max(1, args.gpus)
    base = vo_streams(0, min(job_streams, 8), n)    # pixels of at most 8 distinct streams, shared by the copies
    sat = [base[t % len(base)] for t in range(max(threads, 1))]
    fps, sec, stats, stage = vo_cpu(ora, sat, threads, warm)
    job = [base[t % len(base)] for t in range(job_streams)]
    fps_job, sec_job, _, _ = vo_cpu(ora, job, min(threads, job_streams), warm)
    fps1, sec1, _, stage1 = vo_cpu(ora, base[:1], 1, warm)
    tot = sum(stage.values()) or 1.0
    line = {
        "impl": "reference", "metric": "tracked frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8+f32+f64", "data": "synthetic",
        "config": vo_config(S, F),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": f"{len(sat)} independent streams (one per usable host thread) x {Fs} frames per step x {args.steps} steps "
                                   f"after {args.warmup} warm-up steps; C++ loop on the CPU restatement of the reference (oracle/vo_cpu.cpp, "
                                   f"-O3 AVX2/FMA; the reference itself cannot be built here)",
                         "same_job": {"streams": job_streams, "threads": min(threads, job_streams), "frames_per_s": fps_job},
                         "one_thread_frames_per_s": fps1,
                         "stage_share": {k: v / tot for k, v in stage.items()},
                         "logical_cpus": os.cpu_count(), "affinity_cpus": affinity, "cgroup_cpu_quota": quota,
                         "streams_lost": int(sum(s["lost"] for s in stats))},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, **arrays) -> None:
    """Writes every array as <out_dir>/<name>.npy in float64.  The poses of one step take 96 bytes per frame, so the frames
    the resident leg keeps in HBM (307 kB each) bound them far below DUMP_LIMIT_BYTES; the check makes sure of it."""
    out = {k: np.asarray(v, np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed {DUMP_LIMIT_BYTES}")
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for k, a in out.items():
        np.save(d / f"{k}.npy", a)


def vo_gpu_leg(ctx, stacked, depths, threads, warm, device_ptr=None, window=8, engine="resident"):
    from ygz_slam_b200 import vo_native
    S, n = stacked.shape[:2]
    kw = dict(warm=warm, threads=threads, details=True, window=window, engine=engine)
    if device_ptr is not None:
        return vo_native.run(ctx, None, depths, KF_POLICY["kf_min_frames"], KF_POLICY["kf_min_rot"], KF_POLICY["kf_min_trans"],
                             device_frames=(device_ptr, S, n), **kw)
    return vo_native.run(ctx, stacked, depths, KF_POLICY["kf_min_frames"], KF_POLICY["kf_min_rot"], KF_POLICY["kf_min_trans"], **kw)


def vo_line(args, rank, world, local_rank):
    """The default workload: C5.  Returns the JSON line dict on rank 0."""
    import torch
    import torch.distributed as dist
    from ygz_slam_b200 import Context, se3, vo_native

    S, F = args.streams, args.frames_per_step
    n = (args.warmup + args.steps) * F
    warm = args.warmup * F
    timed = n - warm
    numa = bind_to_gpu_numa(local_rank) if not args.no_numa_bind else {"bound": False, "note": "--no-numa-bind"}
    data = vo_streams(S * rank, S, n)
    stacked = vo_native.stack_pinned([d[0] for d in data])
    depths = [d[1] for d in data]
    # host threads (= ygzb contexts = CUDA streams): every thread drives a latency-bound chain of kernels for its streams and the
    # chains of different threads overlap on the GPU.  Measured on one B200 with 32 hardware work queues (see the top of this
    # file), 8 streams: 4 / 8 threads -> 27.4k / 29.9k frames/s; 16 streams: 8 / 16 threads -> 36.6k / 38.8k; 32 streams: 8 / 16
    # threads -> 41.0k / 40.1k.  Default: one thread per stream, at most 8, and no more than the CPUs this rank may use.
    if args.vo_threads > 0:
        threads = max(1, min(args.vo_threads, S))
    else:
        threads = max(1, min(S, 8, max(2, usable_threads()[0] // max(world, 1))))
    # the engine threads spin in their one synchronisation per round; when the threads of all ranks outnumber the CPUs this job
    # may use (a small cgroup quota under an 8-GPU run), they sleep on a blocking event instead
    _, _, quota = usable_threads()
    cpus = int(min(os.cpu_count() or 1, quota if quota else 1e9))   # what the whole job (all ranks) may use: all CPUs or the cgroup quota
    blocking = {"on": True, "off": False}.get(args.vo_sync, world * (threads + 1) > cpus)
    os.environ["YGZ_VO_BLOCKING_SYNC"] = "1" if blocking else "0"
    ctx = Context(local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def check(traj, stats):
        lost = sum(s["lost"] for s in stats)
        errs = [float(np.linalg.norm(se3.se3_log(se3.mul(traj[s, -1], se3.inv(data[s][2][-1]))))) for s in range(S)]
        return lost, max(errs)

    # ---- resident leg (value): all frames in HBM before the timed region; device-timed --------------------------------
    dev = torch.empty((S, n, H, W), dtype=torch.uint8, device="cuda")
    dev.copy_(torch.from_numpy(stacked), non_blocking=True)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    traj_r, stats_r, sec_r, det_r = vo_gpu_leg(ctx, stacked, depths, threads, warm, device_ptr=dev.data_ptr(), window=args.vo_window)
    barrier()
    # ---- e2e leg: host frames through the C ABI, H2D + D2H inside the timed region ------------------------------------
    traj_e, stats_e, sec_e, det_e = vo_gpu_leg(ctx, stacked, depths, threads, warm, window=args.vo_window)
    barrier()
    # Guard against a rare slow FIRST leg (seen in 2 of ~40 runs: the whole first leg of the process, warm-up included, ran ~5x
    # slower than the e2e leg that follows it on the same frames; no throttle reason, clocks at max): the resident leg cannot be
    # slower than the e2e leg, which does the same work plus the uploads.  Like a throttled run it is re-measured ONCE, and both
    # figures are reported.
    remeasured = None
    redo = 1.0 if det_r["device_ms"] > 1.5 * sec_e * 1e3 else 0.0
    if world > 1:
        flag = torch.tensor([redo], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        redo = float(flag[0])
    if redo:
        first_ms = det_r["device_ms"]
        barrier()
        traj_r, stats_r, sec_r, det_r = vo_gpu_leg(ctx, stacked, depths, threads, warm, device_ptr=dev.data_ptr(), window=args.vo_window)
        barrier()
        remeasured = {"first_resident_ms": first_ms, "second_resident_ms": det_r["device_ms"], "e2e_ms": sec_e * 1e3,
                      "reason": "resident leg slower than 1.5x the e2e leg of the same frames"}
    if args.dump_outputs and rank == 0:
        # what the timed (resident) leg returned: the poses of its last step, and the per-stream counters of the run
        dump_outputs(args.dump_outputs, poses=traj_r[:, n - F:], tracking_stats=[list(s.values()) for s in stats_r])
    # diagnostics (untimed legs of the same streams): one frame per stream in flight (the latency mode of the engine) and
    # the per-stage C-ABI path of round 1 (one blocking call per stage and lock-step frame)
    diag = {}
    if world == 1 and not args.no_secondary:
        for name, kw in (("window_1", dict(window=1)), ("per_stage_calls", dict(engine="stages"))):
            try:
                _, st_d, sec_d, _ = vo_gpu_leg(ctx, stacked, depths, threads, warm, **kw)
                diag[name] = {"tracked_frames_per_s_e2e": S * timed / sec_d, "streams_lost": int(sum(s_["lost"] for s_ in st_d))}
            except Exception as e:  # noqa: BLE001
                diag[name] = {"error": repr(e)}
    clocks = sampler.stop()
    del dev
    lost, err = check(traj_e, stats_e)
    ms_resident, ms_e2e = det_r["device_ms"], sec_e * 1e3

    # ---- per-kernel shares: a short profiled pass on one context (CUDA events around every launch) --------------------
    n_prof = min(n, warm + 2 * F)
    ctx.profile(True)
    _, stats_p, _, _ = vo_gpu_leg(ctx, stacked[:, :n_prof], depths, 1, 0, window=args.vo_window)
    prof = ctx.profile_read()
    ctx.profile(False)

    sharded = None
    if world > 1 and S % world == 0:
        # BASELINE's sentence "8 streams sharded across the GPUs": the same 8 streams of the whole job, 8 / N per GPU
        Ss = S // world
        sh_data = vo_streams(Ss * rank, Ss, n)
        sh_stacked = vo_native.stack_pinned([d[0] for d in sh_data])
        barrier()
        _, st_s, sec_s, det_s = vo_gpu_leg(ctx, sh_stacked, [d[1] for d in sh_data], max(1, min(threads, Ss)), warm, window=args.vo_window)
        barrier()
        t = torch.tensor([sec_s * 1e3, float(sum(s["lost"] for s in st_s))], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sharded = {"streams_total": S, "streams_per_gpu": Ss, "tracked_frames_per_s_e2e": S * timed / (float(t[0]) * 1e-3),
                   "ms_per_step": float(t[0]) / args.steps, "streams_lost_max": int(t[1]), "scaling": "strong"}

    per_rank = None
    if world > 1:
        from ygz_slam_b200 import dist as ydist
        rec = ydist.make_record(rank, S * timed, sum(s["inliers"] for s in stats_e), lost,
                                [ms_e2e, float(numa.get("numa_node", -1)), float(numa.get("cpus_bound", 0)), 1, 0, 0, 0], ms_resident)
        table, _, _ = ydist.gather_records([rec], world, device=torch.device("cuda", local_rank))
        per_rank = [{"rank": int(r[0]), "frames": int(r[1]), "device_ms": float(r[11]), "e2e_ms": float(r[4]), "numa_node": int(r[5]),
                     "cpus_bound": int(r[6])} for r in table]
        t = torch.tensor([ms_resident, ms_e2e, float(lost), err], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_resident, ms_e2e, lost, err = t.tolist()

    line = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        value = world * S * timed / (ms_resident * 1e-3)
        e2e = world * S * timed / (ms_e2e * 1e-3)
        total_ms = sum(v[0] for v in prof.values()) or 1.0
        shares = {k: {"ms_per_launch": v[0] / max(v[1], 1), "launches": v[1], "share": v[0] / total_ms} for k, v in prof.items() if v[1]}
        dom = max(shares, key=lambda k: shares[k]["share"]) if shares else None
        # algorithmic (minimum unique HBM) bytes of the stages of the profiled pass -- DESIGN.md section 4 / SURVEY 8d
        agg = {k: sum(s[k] for s in stats_p) for k in stats_p[0]}
        prof_frames = S * n_prof
        slot3 = sum(((W + (1 << L) - 1) >> L) * ((H + (1 << L) - 1) >> L) for L in range(3))   # 3-level pyramid bytes
        alg = {
            "local_ba": 24.0 * agg["ba_obs"] + 48.0 * agg["ba_pts"] + 96.0 * agg["ba_kfs"],          # obs in, landmarks in+out, poses in+out
            "sparse_align": (prof_frames - S) * (2.0 * slot3) + 25.0 * (agg["candidates"] / 3.0),     # ref + cur pyramid once, ref features
            "project_align": 25.0 * agg["candidates"] + agg["candidates"] * (100 + 81.0),            # candidate record + the two patches' pixels
            "pose_only": 40.0 * agg["projected"],
            "pyrdown": prof_frames * float(slot3), "fast_cells": agg["keyframes"] * float(slot3),
            "describe": agg["keyframes"] * 1244 * (961 + 32.0),
        }
        roof = []
        for k, sh in sorted(shares.items(), key=lambda kv: -kv[1]["share"]):
            if not alg.get(k):
                continue
            dur = sh["ms_per_launch"] * sh["launches"] * 1e-3
            ach = alg[k] / dur / 1e9
            roof.append({"kernel": k, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                         "share_of_step": sh["share"], "us_per_launch": sh["ms_per_launch"] * 1e3, "launches_profiled": sh["launches"],
                         "algorithmic_bytes_per_launch": alg[k] / sh["launches"]})
        main_roof = next((dict(r) for r in roof if r["kernel"] == dom), dict(roof[0]) if roof else None)
        if main_roof is not None:
            main_roof["peak_source"] = peak_src
            try:
                tr = json.loads((ROOT / "profiles" / "r2_dram_traffic.json").read_text()).get(main_roof["kernel"], {})
                if tr.get("dram_bytes_per_problem") and main_roof["kernel"] == "local_ba":
                    # captured per problem (= per cluster); a launch of the profiled pass carries agg["ba"] / launches problems
                    main_roof["traffic"] = tr["dram_bytes_per_problem"] * agg["ba"] / max(shares["local_ba"]["launches"], 1)
                    main_roof["traffic_source"] = tr.get("source")
            except Exception:  # noqa: BLE001
                pass
            if main_roof["kernel"] == "local_ba" and "local_ba" in shares:
                dur = shares["local_ba"]["ms_per_launch"] * shares["local_ba"]["launches"] * 1e-3
                main_roof["fp64"] = {
                    "achieved_gflops": agg["ba_flops"] / dur / 1e9, "nominal_peak_gflops": 40000.0,
                    "frac_of_nominal": agg["ba_flops"] / dur / 1e9 / 40000.0,
                    "ms_per_lm_trial_per_launch": shares["local_ba"]["ms_per_launch"] / max(agg["ba_trials"] / max(agg["ba"], 1), 1),
                    "note": "FLOP model of SURVEY 8d (per LM trial 300 n_obs + sum_j(216 k_j^2 + 108 k_j + 50) + dim^3/3); the BA reduce is FP64 "
                            "ALU / latency bound, not HBM bound -- no FP64 peak is in MEASURED_PEAKS.json, 40 TFLOP/s is the nominal B200 figure"}

        cpu = None
        extra = None
        if world == 1:
            try:
                from oracle.pyoracle import Oracle
                ora = Oracle(native=True)
                thr, affinity, quota = usable_threads()
                ncpu = min(n, 3 + 30)
                sample = [(d[0][:ncpu], d[1], d[2][:ncpu]) for d in data]
                fps1, sec1, st1, stage1 = vo_cpu(ora, sample[:2], 1, 3)
                fpsS, secS, _, _ = vo_cpu(ora, sample, min(thr, S), 3)
                tot = sum(stage1.values()) or 1.0
                cpu = {"value": fps1, "unit": "frames/s", "cores": 1, "kind": "port",
                       "sample": f"frames 3..{ncpu - 1} of 2 of the {S} streams through the same loop in C++ on the CPU oracle (oracle/vo_cpu.cpp, "
                                 f"-O3 AVX2/FMA), single thread like the reference's own code ({sec1:.1f} s of CPU work)",
                       "one_thread_per_stream": {"threads": min(thr, S), "streams": S, "frames_per_s": fpsS, "seconds": secS},
                       "stage_share_1_thread": {k: v / tot for k, v in stage1.items()},
                       "logical_cpus": os.cpu_count(), "affinity_cpus": affinity, "cgroup_cpu_quota": quota}
                try:
                    cpu["opencv_owned_stages"] = opencv_owned_stages(ora)
                except Exception as e:  # noqa: BLE001
                    cpu["opencv_owned_stages"] = {"error": repr(e)}
            except Exception as e:  # noqa: BLE001 -- the headline line must still be printed
                cpu = {"error": repr(e)}
            if not args.no_secondary:
                c8 = None
                try:
                    c8 = Context(local_rank, n_levels=LEVELS)   # C3 runs the 4-level alignment of BASELINE configs[2]
                    extra = secondary_workloads(c8)
                except Exception as e:  # noqa: BLE001
                    extra = {"error": repr(e)}
                finally:
                    if c8 is not None:
                        c8.close()
        line = {
            "metric": "tracked frames/sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_resident / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8+f32+f64", "data": "synthetic",
            "config": vo_config(S, F),
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": (det_e["h2d_image_bytes"] + det_e["h2d_other_bytes"]) / args.steps,
                    "d2h_bytes_per_step": det_e["d2h_bytes"] / args.steps, "ms_per_step": ms_e2e / args.steps,
                    "h2d_image_bytes_per_step": det_e["h2d_image_bytes"] / args.steps,
                    "timing": "wall clock between device synchronisations (host bookkeeping and several CUDA streams are part of the step)"},
            "gpu_launches": int(det_r["gpu_launches"]),
            "resident_remeasured": remeasured,
            # serialised kernel time of the profiled pass (CUDA events around every launch, one context) scaled to the timed region,
            # over the timed wall: > 1 means kernels of several CUDA streams overlapped
            "gpu_busy": {"kernel_ms_per_frame_serialised": total_ms / prof_frames,
                         "kernel_time_over_wall_resident": (total_ms / prof_frames) * S * timed / ms_resident,
                         "kernel_time_over_wall_e2e": (total_ms / prof_frames) * S * timed / ms_e2e},
            "clocks": clocks,
            "roofline": main_roof, "roofline_kernels": roof, "kernel_shares": shares,
            "cpu_baseline": cpu,
            "engine": {"host_threads_per_gpu": threads, "frames_in_flight_per_stream": args.vo_window, "blocking_sync": bool(blocking),
                       "usable_cpus": cpus,
                       "note": "device-resident engine (ygzb_tracker_*: local map, candidate projection, key-frame insertion, BA assembly on "
                               "the device), host loop in C++ (ygz_slam_b200/host/vo_driver.cpp), one ygzb context (CUDA stream) per host "
                               "thread; a round enqueues for every stream the frames up to the first possible key-frame; resident leg wall "
                               "ms %.2f vs device ms %.2f" % (sec_r * 1e3, det_r["device_ms"]),
                       "other_modes": diag},
            "tracking": {"streams_lost": int(lost), "final_pose_error_vs_gt_max": err,
                         "keyframes": int(sum(s["keyframes"] for s in stats_e)), "local_bas": int(sum(s["ba"] for s in stats_e)),
                         "candidates_per_frame": sum(s["candidates"] for s in stats_e) / (S * n),
                         "inliers_per_frame": sum(s["inliers"] for s in stats_e) / (S * n)},
            "sharded_8_streams": sharded,
            "numa": numa,
            "secondary_workloads": extra,
            "per_rank": per_rank,
        }
    ctx.close()
    return line

def extract_match_line(args, rank, world, local_rank, with_secondary=True):
    """BASELINE configs[1] (C2): FAST+ORB extract + brute-force Hamming match over a batch of frames (the round-1 headline,
    now `--workload extract_match` and a secondary record of the default run).  Returns the JSON line dict on rank 0."""
    import torch
    import torch.distributed as dist
    from ygz_slam_b200 import Context

    line = None
    if not getattr(args, "no_numa_bind", False):
        bind_to_gpu_numa(local_rank)
    B = args.batch
    ctx = Context(local_rank, n_levels=LEVELS)
    fr = ctx.frames(B)
    frames = make_frames(B, seed=rank)             # every rank owns an independent stream of frames
    pinned = torch.empty((B, H, W), dtype=torch.uint8).pin_memory()
    pinned.numpy()[:] = frames
    slots = np.arange(B, dtype=np.int32)
    nxt = (slots + 1) % B
    ext = torch.cuda.ExternalStream(ctx.stream, device=local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def resident_step():
        fr.build_pyramid(0, B)
        fr.detect(slots, fetch=False)
        fr.match(slots, nxt, True, fetch=False)

    d2h_bytes = [0]

    # ---- resident leg (value) -------------------------------------------------------------------
    fr.upload_raw(pinned.data_ptr(), B, 1, FRAME_BYTES)   # level 0 resident before the timed region
    ctx.synchronize()
    for _ in range(args.warmup):
        resident_step()
    ctx.synchronize()
    launches0 = ctx.launch_count
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ext):
        ev0.record()
    for _ in range(args.steps):
        resident_step()
    with torch.cuda.stream(ext):
        ev1.record()
    barrier()
    ms_resident = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - launches0

    # ---- e2e leg ----------------------------------------------------------------------------------
    # The public API is synchronous per call (results are back in host memory when it returns), so a
    # user overlaps the PCIe copies of one batch with the kernels of another the way the header says:
    # one context per host thread.  `--e2e-contexts` threads each own a context + slot storage + pinned
    # batch and run whole steps; the timed region covers all of them (wall clock bracketed by barriers,
    # because the work spans several streams).
    n_thr = max(1, args.e2e_contexts)
    while B % n_thr:
        n_thr -= 1
    # every step's batch is split evenly over the contexts (sub-batch i = frames [i*Bs, (i+1)*Bs), each frame matched
    # against its successor, cyclic inside the sub-batch), so all K steps flow through all contexts and the copies of
    # one sub-batch overlap the kernels of the others in steady state
    Bs = B // n_thr
    slots_s = np.arange(Bs, dtype=np.int32)
    nxt_s = (slots_s + 1) % Bs
    workers = []
    for t in range(n_thr):
        c2, f2 = (ctx, fr) if t == 0 else (None, None)
        if c2 is None:
            c2 = Context(local_rank, n_levels=LEVELS)
            f2 = c2.frames(Bs)
        p2 = torch.empty((Bs, H, W), dtype=torch.uint8).pin_memory()
        p2.copy_(pinned[t * Bs:(t + 1) * Bs])
        workers.append((c2, f2, p2))

    call_s = [0.0, 0.0, 0.0, 0]   # worker 0: seconds inside upload / detect / match, calls (diagnostic)

    def e2e_step_on(w):
        c_, f_, p_ = w
        t_a = time.perf_counter()
        f_.upload_raw(p_.data_ptr(), Bs, 1, FRAME_BYTES)
        t_b = time.perf_counter()
        off, _ = f_.detect_packed(slots_s)
        t_c = time.perf_counter()
        qoff, _, _ = f_.match_packed(slots_s, nxt_s, True)
        if w is workers[0]:
            t_d = time.perf_counter()
            call_s[0] += t_b - t_a; call_s[1] += t_c - t_b; call_s[2] += t_d - t_c; call_s[3] += 1
        nf = int(off[-1])
        return nf, nf * (4 + 4 + 1 + 4 + 4 + 32 + 4) + (Bs + 1) * 4 + int(qoff[-1]) * 8 + (Bs + 1) * 4

    def e2e_run(n_steps):
        res = [None] * n_thr

        def work(t):
            out = None
            for _ in range(n_steps):
                out = e2e_step_on(workers[t])
            res[t] = out

        ths = [threading.Thread(target=work, args=(t,)) for t in range(n_thr)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        return sum(r[0] for r in res), sum(r[1] for r in res)

    e2e_run(3)
    call_s[:] = [0.0, 0.0, 0.0, 0]   # the warm-up steps allocate pinned result buffers: keep them out of the per-call diagnostics
    barrier()
    t0 = time.perf_counter()
    nfeat, d2h = e2e_run(args.steps)
    torch.cuda.synchronize()
    ms_e2e_py = (time.perf_counter() - t0) * 1e3
    barrier()
    # the same leg driven by native host threads (ygz_slam_b200/host/e2e_driver.cpp): identical C-ABI calls and buffers
    # without the interpreter lock between them -- this is the e2e figure; the Python-threads figure stays as a diagnostic
    ms_e2e, e2e_how = ms_e2e_py, "python threads"
    try:
        import ctypes as C_
        from ygz_slam_b200 import build as ybuild
        vlib = C_.CDLL(str(ybuild.VO_LIB))
        vlib.ygz_e2e_run.restype = C_.c_int
        vlib.ygz_e2e_run.argtypes = [C_.c_int, C_.c_void_p, C_.c_int, C_.c_int, C_.c_void_p, C_.c_size_t, C_.c_int, C_.c_int, C_.c_void_p,
                                     C_.c_void_p]
        sec = C_.c_double(0.0)
        totals = (C_.c_int64 * 4)()
        rc = vlib.ygz_e2e_run(local_rank, C_.byref(ctx.params), n_thr, Bs, pinned.data_ptr(), FRAME_BYTES, max(args.warmup, 3), args.steps,
                              C_.byref(sec), totals)
        if rc != 0:
            raise RuntimeError(f"ygz_e2e_run rc={rc}")
        barrier()
        ms_e2e, e2e_how = sec.value * 1e3, "native host threads (host/e2e_driver.cpp)"
        if int(totals[0]) != int(nfeat):
            raise RuntimeError(f"native e2e leg found {int(totals[0])} features per step, the Python leg {int(nfeat)}")
        d2h = int(totals[1])
        e2e_launches = int(totals[2])
    except Exception as e:  # noqa: BLE001 -- fall back to the Python-threads figure, say so
        e2e_how = f"python threads (native driver unavailable: {e!r})"
        e2e_launches = None
    d2h_bytes[0] = d2h
    clocks = sampler.stop()
    # diagnostics (untimed): what the PCIe link gives this process, and where worker 0 spent its wall time
    e2e_diag = {"driver": e2e_how, "python_threads_frames_per_s": world * B * args.steps / (ms_e2e_py * 1e-3),
                "gpu_launches_in_e2e_region": e2e_launches,
                "python_worker0_ms_per_call": {k: 1e3 * call_s[i] / max(call_s[3], 1) for i, k in enumerate(("upload", "detect_packed", "match_packed"))}}
    try:
        dev_buf = torch.empty_like(pinned, device="cuda")
        back = torch.empty_like(pinned).pin_memory()
        for name, dst, src in (("h2d_gbs", dev_buf, pinned), ("d2h_gbs", back, dev_buf)):
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(4):
                dst.copy_(src, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            e2e_diag[name] = 4 * pinned.numel() / (e0.elapsed_time(e1) * 1e-3) / 1e9
        ctx.synchronize()
        t_u = time.perf_counter()
        for _ in range(4):
            fr.upload_raw(pinned.data_ptr(), B, 1, FRAME_BYTES)
        ctx.synchronize()
        e2e_diag["upload_api_gbs"] = 4 * pinned.numel() / (time.perf_counter() - t_u) / 1e9
        e2e_diag["e2e_cap_frames_per_s_from_h2d"] = e2e_diag["h2d_gbs"] * 1e9 / FRAME_BYTES * world
        del dev_buf, back
    except Exception as e:  # noqa: BLE001
        e2e_diag["error"] = repr(e)

    # ---- per-kernel shares (CUDA events around every launch; separate pass so the timed legs stay clean)
    ctx.profile(True)
    for _ in range(max(3, args.steps // 2)):
        resident_step()
    prof = ctx.profile_read()
    ctx.profile(False)
    n_prof_steps = max(3, args.steps // 2)

    per_rank = None
    if world > 1:
        # per-rank result records gathered over NCCL (the only collective of the job: results, not pixels)
        from ygz_slam_b200 import dist as ydist
        rec = ydist.make_record(rank, B * args.steps, nfeat, 0, [0, 0, 0, 1, 0, 0, 0], ms_resident)
        table, _, _ = ydist.gather_records([rec], world, device=torch.device("cuda", local_rank))
        per_rank = [{"rank": int(r[0]), "frames": int(r[1]), "device_ms": float(r[11])} for r in table]
        t = torch.tensor([ms_resident, ms_e2e], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_resident, ms_e2e = t.tolist()

    if rank == 0:
        peak, peak_src = measured_peaks()
        value = world * B * args.steps / (ms_resident * 1e-3)
        e2e = world * B * args.steps / (ms_e2e * 1e-3)
        total_ms = sum(v[0] for v in prof.values()) or 1.0
        shares = {k: {"ms_per_launch": v[0] / max(v[1], 1), "launches_per_step": v[1] / n_prof_steps,
                      "share": v[0] / total_ms} for k, v in prof.items() if v[1]}
        kpf = nfeat / B
        alg_bytes = {  # ALGORITHMIC bytes per launch (DESIGN.md section 4)
            "match": B * (32 * 2 * kpf + 8 * kpf),
            "fast_cells": B * PYR_BYTES,
            "pyrdown": None, "describe": B * kpf * (961 + 32), "merge_cells": None,
        }
        dom = max(shares, key=lambda k: shares[k]["share"])
        # measured DRAM bytes per frame of each kernel from the committed `ncu --set full` captures (profiles/), scaled
        # to this launch's frame count (null when the capture is missing)
        try:
            ncu_traffic = json.loads((ROOT / "profiles" / "r1_dram_traffic.json").read_text())
        except Exception:  # noqa: BLE001
            ncu_traffic = {}
        ncu_key = {"match": "match_kernel", "fast_cells": "fast_cells", "describe": "describe_store"}
        roof = []
        for k in ("match", "fast_cells", "describe"):
            if k in shares and alg_bytes.get(k):
                dur = shares[k]["ms_per_launch"] * 1e-3
                ach = alg_bytes[k] / dur / 1e9
                tr = ncu_traffic.get(ncu_key[k], {}).get("dram_bytes_per_frame")
                roof.append({"kernel": k, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                             "frac": ach / peak, "traffic": (tr * B if tr else None),
                             "traffic_source": "profiles/r1_dram_traffic.json (dram__bytes_read+write per frame from ncu --set full) x frames per launch" if tr else None,
                             "share_of_step": shares[k]["share"],
                             "us_per_launch": dur * 1e6, "algorithmic_bytes_per_launch": alg_bytes[k]})
        if "pyrdown" in shares:   # the one kernel family of the step that is HBM-bound by nature: all its launches together
            dur = shares["pyrdown"]["ms_per_launch"] * shares["pyrdown"]["launches_per_step"] * 1e-3
            tr = ncu_traffic.get("pyrdown_stream", {}).get("dram_bytes_per_frame")
            roof.append({"kernel": "pyrdown (all launches of a step)", "bound": "hbm", "achieved": 409600.0 * B / dur / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": 409600.0 * B / dur / 1e9 / peak,
                         "traffic": (tr * B if tr else None),
                         "traffic_source": "largest launch only (level 0 -> 1), profiles/r1_dram_traffic.json" if tr else None,
                         "share_of_step": shares["pyrdown"]["share"], "us_per_launch": dur * 1e6 / shares["pyrdown"]["launches_per_step"],
                         "algorithmic_bytes_per_launch": 409600.0 * B / shares["pyrdown"]["launches_per_step"]})
        main_roof = next((r for r in roof if r["kernel"] == dom), roof[0] if roof else None)
        if main_roof is not None:
            main_roof = dict(main_roof)
            main_roof["peak_source"] = peak_src
            if dom == "match":
                # the matcher is bound by the integer POPC pipe, not by HBM: report that roofline beside it
                sm_mhz = clocks.get("sm_mhz") or 1965.0
                popc_peak = 148 * 16 * sm_mhz * 1e6               # POPC lanes/clk/SM x SMs x clock
                pairs_per_s = B * kpf * kpf / (shares["match"]["ms_per_launch"] * 1e-3)
                main_roof["popc_pipe"] = {
                    "algorithmic_gpopc_s": 8 * pairs_per_s / 1e9,     # SURVEY 8d counts 8 POPC per descriptor pair
                    "executed_popc_per_pair": 5,                      # carry-save adders fold the 8 words into 5 POPC
                    "executed_gpopc_s": 5 * pairs_per_s / 1e9, "peak_gpopc_s": popc_peak / 1e9,
                    "pipe_utilisation": 5 * pairs_per_s / popc_peak,
                    "note": "peak = 148 SMs x 16 POPC/clk/SM (measured, profiles/r1_microbench_int_pipes.txt) x sampled SM clock"}

        # ---- bounded CPU baseline (rank 0, N=1 only) ----------------------------------------------
        cpu = None
        if world == 1:
            from oracle.pyoracle import Oracle
            ora = Oracle(native=True)
            ns = args.cpu_sample
            cpu_run(ora, frames, 2, 1)
            dt, _ = cpu_run(ora, frames, ns, 1)
            cpu = {"value": ns / dt, "unit": "frames/s", "cores": 1, "kind": "port",
                   "sample": f"{ns} frames of the same batch (pyramid+Detect+cross-checked BF match), oracle -O3 AVX2/FMA "
                             f"build, single thread like the reference's own code; host has {os.cpu_count()} logical CPUs"}

        extra = None
        if world == 1 and with_secondary:
            try:
                extra = secondary_workloads(ctx)
            except Exception as e:  # noqa: BLE001 -- the headline line must still be printed
                extra = {"error": repr(e)}

        line = {
            "metric": "tracked frames/sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_resident / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(B, "one batch of independent frames per GPU per step"),
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": B * FRAME_BYTES, "d2h_bytes_per_step": d2h_bytes[0],
                    "ms_per_step": ms_e2e / args.steps, "host_threads": n_thr, "frames_per_context_per_step": Bs, "diag": e2e_diag,
                    "timing": "wall clock between device synchronisations (the leg spans several streams)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": main_roof,
            "roofline_kernels": roof,
            "kernel_shares": shares,
            "cpu_baseline": cpu,
            "keypoints_per_frame": kpf,
            "secondary_workloads": extra,
            "per_rank": per_rank,
        }
    for c_, f_, _ in workers[1:]:
        f_.close()
        c_.close()
    fr.close()
    ctx.close()
    return line if rank == 0 else None



def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="vo", choices=["vo", "extract_match"],
                    help="vo = BASELINE metric (tracked frames/sec, configs[4] C5: 8 streams per GPU through the full tracking loop; "
                         "the headline); extract_match = configs[1] C2 (FAST+ORB extract + BF match)")
    ap.add_argument("--streams", type=int, default=8, help="vo: independent streams per GPU")
    ap.add_argument("--frames-per-step", type=int, default=10, help="vo: frames per stream and step")
    ap.add_argument("--vo-threads", type=int, default=0,
                    help="vo: host threads (= ygzb contexts = CUDA streams) per GPU; 0 = one per stream, capped by the usable CPUs per rank")
    ap.add_argument("--vo-window", type=int, default=8, help="vo: frames of one stream that may be in flight per round (1 = latency mode)")
    ap.add_argument("--vo-sync", default="auto", choices=["auto", "on", "off"],
                    help="vo: blocking (sleeping) synchronisation of the engine threads; auto = only when they outnumber the usable CPUs")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the CPUs local to its GPU")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary workloads (C2, C3, C4) of the N=1 run")
    ap.add_argument("--batch", type=int, default=512, help="extract_match: frames per step per GPU")
    ap.add_argument("--cpu-sample", type=int, default=48, help="extract_match: frames of the bounded cpu_baseline sample")
    ap.add_argument("--e2e-contexts", type=int, default=8,
                    help="extract_match: host threads (one ygzb context = one stream each) used by the e2e leg so that the H2D "
                         "copy of one batch overlaps the kernels of another")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="vo: after the timed steps, write what the timed leg computed as DIR/<name>.npy (float64): poses.npy = "
                         "(streams, frames per step, 3, 4) camera poses T_cw of the last step, tracking_stats.npy = (streams, 12) "
                         "per-stream counters (lost, keyframes, ba, candidates, projected, inliers, ba_obs, ba_pts, ba_kfs, "
                         "ba_trials, ba_iters, ba_flops); rank 0's streams")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "vo"):
        ap.error("--dump-outputs writes the outputs of the GPU path of the vo workload")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if args.workload == "vo":
            run_reference_vo(args, rank, world)
        else:
            run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    if args.workload == "vo":
        line = vo_line(args, rank, world, local_rank)
        if rank == 0 and world == 1 and not args.no_secondary:
            # BASELINE configs[1] (C2) as a secondary record: a short run of the round-1 headline
            try:
                a2 = argparse.Namespace(**vars(args))
                a2.steps, a2.warmup = 5, 3
                c2 = extract_match_line(a2, rank, world, local_rank, with_secondary=False)
                keep = ("value", "unit", "ms_per_step", "e2e", "roofline", "cpu_baseline", "keypoints_per_frame", "config", "gpu_launches")
                line.setdefault("secondary_workloads", {})
                if not isinstance(line["secondary_workloads"], dict):
                    line["secondary_workloads"] = {"note": line["secondary_workloads"]}
                line["secondary_workloads"]["c2_extract_match_512_frames"] = {k: c2[k] for k in keep if k in c2}
            except Exception as e:  # noqa: BLE001
                line.setdefault("secondary_workloads", {})
                if isinstance(line["secondary_workloads"], dict):
                    line["secondary_workloads"]["c2_error"] = repr(e)
    else:
        line = extract_match_line(args, rank, world, local_rank)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
