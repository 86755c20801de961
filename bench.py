#!/usr/bin/env python
"""bench.py — RegisterFrame throughput of the B200-native CT-ICP engine on BASELINE.json's metric.

A "step" is one cticp RegisterFrame of one synthetic KITTI-shape 64-beam scan (HDL-64E ring table, ~130k returns of the
"suburb" scene: F ~ 12k frame points, K ~ 2.6k keypoints) with the driving options of BASELINE.json configs[1] (solver GN,
5 ICP iterations, map voxel 1.0 m / 20 pts, voxel_size 0.5, sample_voxel_size 1.5). Steps are consecutive frames of ONE
odometry run: the first `--preroll` frames (the reference's start-up regime, init_num_frames = 20) and the W warm-up
frames are registered untimed.

  value       scans/s with the packed scans already resident in HBM (cticp_odometry_register_staged), timed per step
              with CUDA events on the engine's stream, L2 flushed (untimed 256 MiB memset) between steps
  e2e         scans/s through cticp_odometry_register_frame with HOST numpy buffers: host packing into pinned memory, H2D
              of the scan, all kernels, the frame verdict (poses / counters / decisions, written by the device into mapped
              pinned memory); wall clock per step incl. the map-update tail
  e2e_dropin  the same call with the reference's full RegistrationSummary contract (src/ct_icp/odometry.cpp:462-486,597):
              corrected_points, all_corrected_points and keypoints are transformed, copied back and assembled into
              caller-owned arrays of 64-byte WPoint3D records inside the timed region
  roofline    k_gn_persistent (all ICP iterations of a frame in one launch: gather + selection + reduce + solve):
              algorithmic bytes per launch / CUDA-event time per launch vs the measured HBM copy bandwidth
  cpu_baseline  the CPU oracle (restatement of the reference's path with the reference's threading) on the same frames
  extra_workloads  configs[2] (driving_config.yaml, solver CERES as a device LM/IRLS loop) and configs[4] (dense 128-beam
              scans, 20 forced GN iterations) measured the same way on fewer frames, each with its own cpu_baseline

`--impl reference` times only the CPU oracle (the reference itself cannot be built offline, see DESIGN.md).
`--dump-outputs DIR` writes what the timed path returned for its last step as DIR/<name>.npy (see dump_outputs); the scans
are seeded, so two builds (or the two arms) run with the same arguments can be compared output for output.
N > 1 (torchrun): every rank registers the same scans with the keypoints sharded rank/world; the JTJ/JTr sums are
exchanged inside the persistent GN kernel over NVLink peer mailboxes ("strong" scaling of one frame's latency). Rank 0
also registers the first frames unsharded and the line carries the sharded-vs-single pose difference.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree it runs from (which may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "scans/sec (RegisterFrame) on 64-beam ~120k-pt clouds"
UNIT = "scans/s"
WORKLOAD = "configs[1]: KITTI-shape 64-beam synthetic scans, CT_ICP_GN point-to-plane, 5 ICP iters, 1xB200"


WORKLOADS = {
    # name: (sensor, description)
    "kitti64_gn": ("HDL64E", WORKLOAD),
    "kitti64_ceres": ("HDL64E", "configs[2]: KITTI-shape 64-beam synthetic scans, driving_config.yaml (solver CERES as device "
                                "LM/IRLS, Cauchy, 5x5 iterations, 900 residuals), 1xB200"),
    "dense128_gn": ("DENSE128", "configs[4]: dense 128-beam ~290k-pt synthetic scans, CT_ICP_GN, 20 ICP iterations forced, "
                                "voxel 0.25 / sample 0.5, 1xB200"),
}
_WORKLOAD = "kitti64_gn"
SCENE_PROFILE = "suburb"


def make_options(b):
    from ct_icp_b200 import _abi as abi
    if _WORKLOAD == "kitti64_ceres":
        o = b.profile("default_driving")
        o.debug_print = 0
        o.neighborhood_strategy.max_num_neighbors = 20
        o.neighborhood_strategy.min_num_neighbors = 10
        m = b.default_map_options()
        m.num_resolutions = 1
        m.resolutions[0].resolution = 0.8
        m.resolutions[0].max_num_points = 30
        m.resolutions[0].min_distance_between_points = 0.1
        m.default_radius = 0.75
        o.map_options = m
        c = o.ct_icp_options
        c.debug_print = 0
        c.num_iters_icp, c.solver, c.max_num_residuals = 5, abi.SOLVER["CERES"], 900
        c.min_number_neighbors = c.max_number_neighbors = 20
        c.threshold_orientation_norm, c.threshold_translation_norm = 0.1, 0.01
        c.loss_function, c.ls_max_num_iters, c.ls_num_threads, c.ls_sigma = abi.LOSS["CAUCHY"], 5, 6, 0.1
        return o
    if _WORKLOAD == "dense128_gn":
        o = b.default_odometry_options()
        o.debug_print = 0
        o.ct_icp_options.solver = abi.SOLVER["GN"]
        o.ct_icp_options.num_iters_icp = 20
        o.ct_icp_options.threshold_orientation_norm = 0.0
        o.ct_icp_options.min_number_neighbors = 10
        o.map_options = b.legacy_map_options(1.0, 20, 0.1)
        o.voxel_size = o.init_voxel_size = 0.25
        o.sample_voxel_size = o.init_sample_voxel_size = 0.5
        return o
    o = b.default_odometry_options()
    o.ct_icp_options.solver = abi.SOLVER["GN"]
    o.ct_icp_options.num_iters_icp = 5
    o.ct_icp_options.min_number_neighbors = 10      # test/regression/regression_config_short_drive.yaml:93
    o.ct_icp_options.max_number_neighbors = 20
    o.ct_icp_options.max_dist_to_plane_ct_icp = 0.3
    o.map_options = b.legacy_map_options(1.0, 20, 0.1)   # size_voxel_map 1.0, 20 pts/voxel, min_distance 0.1
    o.voxel_size = 0.5
    o.sample_voxel_size = 1.5
    o.max_distance = 100.0
    o.debug_print = 0
    o.ct_icp_options.debug_print = 0
    return o


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled DURING the timed region (B200_PROFILING.md's clocks line).

    In-process NVML (pynvml) from a daemon thread every 20 ms (the timed regions are only tens of ms long; at 5 ms the queries began to show in the step times) — two cheap queries per sample, no child process next
    to the HOST-timed end-to-end steps; `nvidia-smi -lms 200` is the fallback (CTICP_BENCH_CLOCKS=smi forces it)."""

    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.sm, self.smax, self.reasons = [], [], set()
        self.mode = os.environ.get("CTICP_BENCH_CLOCKS", "nvml")
        self.stop_flag = threading.Event()
        self.thread = None
        self.proc = None

    def _nvml_loop(self, nv, handle):
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(handle))
                for name, mask in self.REASONS.items():
                    if bits & mask:
                        self.reasons.add(name)
            except Exception:
                pass
            self.stop_flag.wait(0.02)

    def _smi_loop(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 7:
                continue
            try:
                self.sm.append(float(f[0]))
                self.smax.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def start(self):
        if self.mode == "nvml":
            try:
                import pynvml as nv
                nv.nvmlInit()
                # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                idx = self.gpu_index
                if vis and all(v.strip().isdigit() for v in vis.split(",")):
                    idx = int(vis.split(",")[self.gpu_index])
                handle = nv.nvmlDeviceGetHandleByIndex(idx)
                self.smax.append(float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM)))
                self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
                self.thread.start()
                return
            except Exception:
                self.mode = "smi"
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._smi_loop, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def stop(self):
        self.stop_flag.set()
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.thread:
            self.thread.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": max(self.smax) if self.smax else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "sampler": self.mode}


_SCENES = {}


def make_scans(n_frames, sensor_name):
    """The workload's seeded scans (same frames for every arm and every pass)."""
    from ct_icp_b200 import synthetic as syn
    if SCENE_PROFILE not in _SCENES:
        _SCENES[SCENE_PROFILE] = syn.UrbanScene(1234, profile=SCENE_PROFILE)
    return syn.make_sequence(n_frames, getattr(syn, sensor_name), seed=1234, scene=_SCENES[SCENE_PROFILE])


def workload_config(workload_text, world, seq, first, count, frame_points, keypoints, iters, preroll):
    """The `config` object of a bench line: identical keys and values for the native and the reference arm."""
    return {"workload": workload_text.replace("1xB200", "%dxB200" % world),
            "scene": "synthetic '%s' scene, %s" % (SCENE_PROFILE, "ct_icp_b200/synthetic.py"),
            "points_per_scan": round(float(np.mean([len(s["xyz"]) for s in seq[first:first + count]])), 1),
            "frame_points": round(frame_points, 1), "keypoints": round(keypoints, 1),
            "icp_iters_per_step": round(iters, 2), "preroll_frames": preroll}


def run_oracle(seq, first_timed, steps, dump_dir=None):
    """CPU oracle over the same frames; returns (scans/s over the timed steps, per-step ms, F, K, iterations per step).
    dump_dir: the outputs of the last timed step are written there."""
    from oracle_lib import oracle
    orc = oracle()
    od = orc.odometry(make_options(orc))
    times, f_sum, k_sum, it_sum = [], 0, 0, 0
    for i, s in enumerate(seq[:first_timed + steps]):
        t0 = time.perf_counter()
        sm = od.RegisterFrame(s["xyz"], s["t"], s["frame_idx"])
        dt = time.perf_counter() - t0
        if not sm.success:
            raise RuntimeError("oracle registration failed at frame %d: %s" % (i, sm.error_message))
        if i >= first_timed:
            times.append(dt * 1e3)
            f_sum += sm.num_corrected_points
            k_sum += sm.num_keypoints
            it_sum += sm.icp_summary.num_iters
    if dump_dir:
        dump_outputs(dump_dir, od, sm)
    n = max(len(times), 1)
    return len(times) / (sum(times) / 1e3), times, f_sum / n, k_sum / n, it_sum / n


def oracle_threads():
    from oracle_lib import oracle as _orc
    return int(make_options(_orc()).ct_icp_options.ls_num_threads)


CPU_SAMPLE_NOTE = ("CPU oracle restating the reference's RegisterFrame with the reference's threading: GN per-keypoint loop "
                   "serial (src/ct_icp/ct_icp.cpp:753), CERES/ROBUST residual assembly and point transforms on ls_num_threads "
                   "OpenMP threads (ct_icp.cpp:561; odometry.cpp:469,480). A PORT, pessimistic against real ct_icp: it keeps "
                   "voxels in std::unordered_map / std::unordered_set and a std::priority_queue of tuples where the reference "
                   "uses tsl::robin_map (oracle/orc_core.h)")


def load_traffic():
    """dram bytes per launch of the GN kernel from the committed ncu capture summary (profiles/), if any."""
    for name in ("r03_gn_persistent_ncu_summary.json", "r02_gn_persistent_ncu_summary.json", "gather_kernel_ncu_summary.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f).get("dram_bytes_per_launch")
        except Exception:
            continue
    return None


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class Dist:
    """torch.distributed plumbing of the N > 1 runs (one process per GPU)."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.dist = None
        self.device = self.local_rank if self.world > 1 else 0

    def init(self):
        import torch
        self.torch = torch
        if self.world > 1:
            import torch.distributed as dist
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def pose_vector(sm):
    return np.array(list(sm.frame.begin_pose.tr) + list(sm.frame.begin_pose.quat) + list(sm.frame.end_pose.tr) +
                    list(sm.frame.end_pose.quat))


# summary.npy, in this order: the RegistrationSummary's counters and decisions (its timings are left out: they differ
# from run to run), then the map size after the step
SUMMARY_FIELDS = ("success", "sample_size", "number_of_residuals", "robust_level", "points_added", "number_of_attempts",
                  "num_corrected_points", "num_all_corrected_points", "num_keypoints", "distance_correction",
                  "relative_distance", "relative_orientation", "ego_orientation", "icp_success", "icp_num_residuals_used",
                  "icp_num_iters", "map_size")
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, od, sm):
    """What a caller of RegisterFrame receives for the frame `sm` summarises (the last one `od` registered), as float64
    DIR/<name>.npy:
      frame, initial_frame   (2, 8): begin and end pose, each tx ty tz qx qy qz qw dest_timestamp
      summary                SUMMARY_FIELDS
      corrected_points, all_corrected_points, keypoints   (n, 8): the summary's point vectors, one WPoint3D per row:
                             raw xyz, timestamp, world xyz, index_frame
    """
    from ct_icp_b200 import _abi as abi

    def frame_rows(f):
        return np.array([list(p.tr) + list(p.quat) + [p.dest_timestamp] for p in (f.begin_pose, f.end_pose)])

    def points(which):
        p = od.points(which)
        return np.column_stack([p["raw"], p["timestamp"], p["world"], p["index_frame"]]).astype(np.float64)

    def summary_value(name):
        if name == "map_size":
            return od.MapSize()
        if name.startswith("icp_"):
            return getattr(sm.icp_summary, name[len("icp_"):])
        return getattr(sm, name)

    out = {
        "frame": frame_rows(sm.frame), "initial_frame": frame_rows(sm.initial_frame),
        "summary": np.array([summary_value(f) for f in SUMMARY_FIELDS], dtype=np.float64),
        "corrected_points": points(abi.POINTS_CORRECTED),
        "all_corrected_points": points(abi.POINTS_ALL_CORRECTED),
        "keypoints": points(abi.POINTS_KEYPOINTS),
    }
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("outputs of %d bytes exceed the dump limit of %d" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_native(eng, D, seq, preroll, W, K, n_roof, with_dropin=True, parity_frames=0, dump_dir=None):
    """All GPU passes of one workload over `seq`. Returns the fields of the bench line (rank 0) — timing is max over ranks.
    dump_dir: rank 0 writes the outputs of pass A's last timed step there."""
    from ct_icp_b200 import _abi as abi
    torch = D.torch
    world, rank, device = D.world, D.rank, D.device
    first = preroll + W
    shard_modes = []

    def make_odometry(sharded=True):
        od = eng.odometry(make_options(eng), device)
        if world > 1 and sharded:
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                import ctypes
                buf = (ctypes.c_char * 128)()
                eng.check(eng.fn("nccl_unique_id")(buf))
                uid = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).cuda()
            D.dist.broadcast(uid, 0)
            od.enable_sharding(bytes(uid.cpu().numpy().tobytes()), rank, world)
            shard_modes.append(od.sharding_mode())
        return od

    # ---- pass A: device-resident input, CUDA-event timing per step ------------------------------------------
    od = make_odometry()
    slots = [od.stage_frame(s["xyz"], s["t"]) for s in seq]
    head_poses = []
    for i in range(first):
        sm = od.RegisterStaged(slots[i], seq[i]["frame_idx"])
        assert sm.success, sm.error_message
        if i < parity_frames:
            head_poses.append(pose_vector(sm))
    od.last_timing()
    D.barrier()
    step_ms, launches, kp_sum, f_sum, iters_sum = [], 0, 0, 0, 0
    for i in range(first, first + K):
        od.flush_l2(256 << 20)
        if D.dist is not None:
            D.barrier()                   # all ranks receive the scan at the same time (untimed)
        od.timer_start()
        sm = od.RegisterStaged(slots[i], seq[i]["frame_idx"])
        ms = od.timer_stop()
        assert sm.success, sm.error_message
        step_ms.append(ms)
        t = od.last_timing()
        launches += t.kernel_launches
        kp_sum += sm.num_keypoints
        f_sum += sm.num_corrected_points
        iters_sum += t.icp_iterations
    D.barrier()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, od, sm)
    total_ms = D.max_over_ranks(float(np.sum(step_ms)))
    out = {"value": K / (total_ms / 1e3), "ms_per_step": total_ms / K, "gpu_launches": launches,
           "frame_points": f_sum / K, "keypoints": kp_sum / K, "iters": iters_sum / K}

    # ---- roofline pass: CUDA events around the GN kernel of each frame (continues pass A's odometry) -------------
    roofline = None
    if n_roof:
        od.set_gather_timing(True)
        g_ms, g_launch, g_kp, g_pts = 0.0, 0, 0, 0
        solve_share = []
        for i in range(first + K, first + K + n_roof):
            od.flush_l2(256 << 20)
            sm = od.RegisterStaged(slots[i], seq[i]["frame_idx"])
            t = od.last_timing()
            if sm.icp_summary.avg_duration_iter > 0:   # clock64 stamps of the solver CTA (k_gn_persistent)
                solve_share.append(sm.icp_summary.avg_duration_solve / sm.icp_summary.avg_duration_iter)
            g_ms += t.gather_ms
            g_launch += t.gather_launches
            g_kp += t.gather_keypoint_iterations
            g_pts += t.gather_stencil_points
        od.set_gather_timing(False)
        stencil = 27        # (2r+1)^3 with r = ceil(0.8 / 1.0) = 1
        alg_bytes = g_kp * (16 + 16 * stencil) + 16 * g_pts          # SURVEY §8d: keypoint + slot probes + map points
        peak, peak_src = measured_peak_gbs()
        if g_launch and g_ms > 0:
            achieved = (alg_bytes / g_launch) / (g_ms / g_launch * 1e-3) / 1e9
            roofline = {"bound": "hbm", "kernel": "k_gn_persistent (all ICP iterations of a frame: gather + selection + reduce + solve)",
                        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": load_traffic(),
                        "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes / g_launch,
                        "us_per_launch": g_ms / g_launch * 1e3, "keypoint_iterations_per_launch": g_kp / g_launch,
                        "us_per_1k_keypoint_iterations": (g_ms * 1e3) / max(g_kp, 1) * 1e3,
                        "mean_stencil_points": g_pts / max(g_kp, 1), "launches_timed": g_launch,
                        "serial_reduce_and_solve_share": float(np.mean(solve_share)) if solve_share else None}
    out["roofline"] = roofline
    od.clear_staged()
    od.close()

    # ---- sharded vs single GPU on the head of the sequence (N > 1: rank 0 re-registers it unsharded) -----------------
    if world > 1 and parity_frames:
        diff = 0.0
        if rank == 0:
            od1 = make_odometry(sharded=False)
            for i in range(parity_frames):
                sm = od1.RegisterFrame(seq[i]["xyz"], seq[i]["t"], seq[i]["frame_idx"])
                assert sm.success, sm.error_message
                diff = max(diff, float(np.abs(pose_vector(sm) - head_poses[i]).max()))
            od1.close()
            assert diff < 1e-6, "sharded and single-GPU poses differ by %g" % diff
        out["sharded_vs_single"] = {"frames": parity_frames, "max_abs_pose_diff": diff,
                                    "what": "begin/end translation (m) and quaternion of the first frames, %d ranks vs 1" % world}

    # ---- pass B: end to end through the C ABI with host buffers ----------------------------------------------
    def e2e_pass(dropin):
        od = make_odometry()
        bufs = None
        if dropin:
            od.set_summary_points(7)
            cap = max(len(s["xyz"]) for s in seq)
            bufs = [np.zeros(cap, dtype=abi.wpoint_dtype()) for _ in range(3)]
        for i in range(first):
            sm = od.RegisterFrame(seq[i]["xyz"], seq[i]["t"], seq[i]["frame_idx"])
            assert sm.success, sm.error_message
            if dropin:
                for w in (1, 2, 0):
                    od.points_into(w, bufs[w])
        od.last_timing()
        D.barrier()
        ms_list, h2d, d2h = [], 0, 0
        for i in range(first, first + K):
            od.flush_l2(256 << 20)
            torch.cuda.synchronize(device)
            od.last_timing()                  # the previous frame's tail has completed
            if D.dist is not None:
                D.barrier()                   # all ranks receive the scan at the same time (untimed)
            t0 = time.perf_counter()
            sm = od.RegisterFrame(seq[i]["xyz"], seq[i]["t"], seq[i]["frame_idx"])
            if dropin:   # all_corrected_points first: it comes back in pieces, assembled while the rest is still copying
                counts = [0, 0, 0]
                for w in (1, 2, 0):
                    counts[w] = od.points_into(w, bufs[w])
            t = od.last_timing()              # waits for the map-update tail of this frame
            ms_list.append((time.perf_counter() - t0) * 1e3)
            assert sm.success, sm.error_message
            if dropin:
                assert counts[1] == len(seq[i]["xyz"]) and counts[0] == sm.num_corrected_points
            h2d += t.h2d_bytes
            d2h += t.d2h_bytes
        D.barrier()
        total = D.max_over_ranks(float(np.sum(ms_list)))
        od.close()
        return {"value": K / (total / 1e3), "unit": UNIT, "ms_per_step": total / K,
                "ms_per_step_median": float(np.median(ms_list)), "ms_per_step_max": float(np.max(ms_list)),
                "h2d_bytes_per_step": h2d / K, "d2h_bytes_per_step": d2h / K}

    out["e2e"] = e2e_pass(False)
    out["e2e"]["timing"] = "wall clock per step incl. host packing and the map-update tail; poses + counters come back"
    if with_dropin:
        out["e2e_dropin"] = e2e_pass(True)
        out["e2e_dropin"]["timing"] = ("as e2e, plus RegistrationSummary's three point vectors (odometry.cpp:462-486,597) "
                                       "transformed, copied to the host and assembled into caller-owned 64-byte WPoint3D arrays")
    out["parallelism"] = "single GPU" if world == 1 else "keypoints sharded x%d, JTJ/JTr summed over ranks once per iteration: %s" % (
        world, "inside the persistent GN kernel over NVLink peer mailboxes (one launch per frame)"
        if shard_modes and min(shard_modes) == 2 else "ncclAllReduce (peer mapping unavailable)")
    return out


def cpu_baseline_for(seq, first, steps, cores, dump_dir=None):
    v, times, f, k, it = run_oracle(seq, first, steps, dump_dir)
    threads = oracle_threads()
    return {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "ms_per_step": float(np.mean(times)),
            "sample": "%d timed frames (after %d untimed) of the same sequence; %s; %d host CPUs on this box"
                      % (steps, first, CPU_SAMPLE_NOTE, cores)}, (f, k, it)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--preroll", type=int, default=20, help="start-up frames registered untimed before the warm-up")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--roofline-frames", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[2] / configs[4] extra workloads")
    ap.add_argument("--workload", default="kitti64_gn", choices=sorted(WORKLOADS),
                    help="kitti64_gn is BASELINE.json's metric configuration (the bench line)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned for its last step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    global _WORKLOAD, WORKLOAD
    _WORKLOAD = args.workload
    sensor_name, WORKLOAD = WORKLOADS[args.workload]

    D = Dist()
    rank, world = D.rank, D.world
    W = max(args.warmup, 3)
    K = args.steps
    cores = os.cpu_count() or 1
    preroll = args.preroll if args.workload != "dense128_gn" else min(args.preroll, 6)
    first = preroll + W

    # ------------------------------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        seq = make_scans(first + K, sensor_name)
        cb, (f, k, it) = cpu_baseline_for(seq, first, K, cores, args.dump_outputs)
        line = {
            "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": K,
            "warmup": W, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(WORKLOAD, args.gpus, seq, first, K, f, k, it, preroll),
            "arm": {"note": "CPU restatement (oracle/) of the reference's RegisterFrame; the reference cannot be built "
                            "offline (Eigen/Ceres/glog/yaml-cpp/robin_map absent)"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------------------------------ native arm
    D.init()
    import ct_icp_b200
    eng = ct_icp_b200.engine()
    n_roof = args.roofline_frames
    seq = make_scans(first + K + n_roof, sensor_name)
    clocks = ClockSampler(D.device)
    D.barrier()
    clocks.start()
    res = run_native(eng, D, seq, preroll, W, K, n_roof, with_dropin=True, parity_frames=6 if world > 1 else 0,
                     dump_dir=args.dump_outputs)
    clock_info = clocks.stop()     # sampled from the start of the device-timed steps to the end of the e2e steps

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline, _ = cpu_baseline_for(seq, first, K, cores)

    # ---- the other single-GPU configs of BASELINE.json, same passes on fewer frames (extra keys of the same line) ----
    extras = None
    if args.workload == "kitti64_gn" and not args.no_extras:
        extras = {}
        plan = {"kitti64_ceres": (args.preroll, 3, 12, 10), "dense128_gn": (6, 3, 6, 2)}
        if world > 1:
            plan.pop("kitti64_ceres")   # N > 1: only the configuration the sweep of BASELINE.json configs[4] is about
        for name, (xp, xw, xk, xcpu) in plan.items():
            _WORKLOAD = name
            xsensor, xtext = WORKLOADS[name]
            xseq = seq if xsensor == sensor_name else make_scans(xp + xw + xk, xsensor)
            try:
                r = run_native(eng, D, xseq, xp, xw, xk, 0, with_dropin=False)
                entry = {"value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "steps": xk,
                         "config": workload_config(xtext, world, xseq, xp + xw, xk, r["frame_points"], r["keypoints"], r["iters"], xp),
                         "e2e": r["e2e"], "gpu_launches": r["gpu_launches"], "cpu_baseline": None}
                if rank == 0 and world == 1 and not args.no_cpu_baseline:
                    entry["cpu_baseline"], _ = cpu_baseline_for(xseq, xp + xw, xcpu, cores)
                extras[name] = entry
            except Exception as e:   # an extra must never cost the headline line
                extras[name] = {"error": "%s: %s" % (type(e).__name__, e)}
        _WORKLOAD = args.workload

    if rank == 0:
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(WORKLOAD, world, seq, first, K, res["frame_points"], res["keypoints"], res["iters"], preroll),
            "arm": {"l2": "flushed between steps (256 MiB memset, untimed)", "parallelism": res["parallelism"],
                    "storage": "fp32 voxel-local map points / keypoints, fp64 arithmetic"},
            "e2e": res["e2e"],
            "e2e_dropin": res.get("e2e_dropin"),
            "gpu_launches": res["gpu_launches"],
            "clocks": clock_info,
            "roofline": res["roofline"],
            "cpu_baseline": cpu_baseline,
        }
        if "sharded_vs_single" in res:
            line["sharded_vs_single"] = res["sharded_vs_single"]
        if extras is not None:
            line["extra_workloads"] = extras
        print(json.dumps(line))
    if D.dist is not None:
        D.dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
