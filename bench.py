#!/usr/bin/env python
"""bench.py -- ICP odometry frames/s on synthetic 64x2048 scans (BASELINE.json metric).

One "step" = one frame of the BASELINE config-2 pipeline: GridSample(voxel 0.3) -> ToTensor ->
ICPFrameToModel (kd-tree local map of 20 frames, point-to-plane Gauss-Newton, geman_mcclure
sigma 0.3, <= 10 alignments, constant-velocity initialisation), on a seeded synthetic stream.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--no-extra] [--no-cpu] [--dump-outputs DIR]

* `value`  : frames/s with every raw scan already resident in HBM; one C-ABI call per frame
             (pls_process_frame_grid_sample) on device pointers; ONE CUDA-event bracket on the library's
             stream around the K timed frames (closed after both of the library's streams have drained).
             `value` is the MEDIAN of 3 such passes (fresh context, W warm-up frames, exactly K timed frames each; all
             three are listed in config.repeats) -- with the driver's --steps 20 one bracket is a 10 ms sample.
* `e2e`    : frames/s through the reference-shaped Python API (Preprocessing[GridSample, ToTensor]
             -> ICPFrameToModel.process_next_frame) from PINNED HOST buffers, host<->device copies
             inside the timed region; the median of 3 passes as well.
* roofline : the kd correspondence kernels of the executed ICP iterations (verify / 1-NN search / lazy 10-NN normals /
             reduction + fused solve), CUDA-event timed inside the library over the timed frames (a second pass, so
             that the event records do not perturb `value`).  `achieved` uses SURVEY.md 8d's algorithmic bytes with
             the candidate counts the kernels themselves count; `lower_bound` is the 44 B / query + 16 B / touched
             map point figure.
* config.extra_workloads : the HBM-sized configurations of BASELINE.json (cfg3 128x2048 projective, cfg5 128x4096
             x 20 iterations projective, cfg4 5 M-point kd map x 131 072 queries), each with ms/frame, the CUDA-event
             time of its dominant kernel, algorithmic bytes and fraction of the measured HBM peak; at N > 1 also
             sharded over the ranks.
* config.sharded_vs_single (N > 1): poses of a forced-sharded run against rank 0's private single-GPU context.
* cpu_baseline / --impl reference: the CPU oracle port of the reference path (oracle/) on the host
             cores, on a bounded sample of the same stream (--impl reference: at most 24 warm-up frames, then K timed frames).
* --dump-outputs DIR: after the timed passes, what the timed call returned for the last timed frame, as DIR/<name>.npy:
             odometry_pose [4,4] float32, odometry_params [6] float32, frame_info [12] float64 (pls_process_frame's
             out_info); the pass whose time is reported.  --impl reference writes odometry_pose [4,4] float64 alone.
             The scans are seeded, so the same arguments give the same inputs on every run and build.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, W, VOXEL = 64, 2048, 0.3
REPEATS = 3   # independent passes behind `value` and behind `e2e` (the median pass is reported, all are listed)
MAX_ALIGN, LM_SIZE, SCHEME, SIGMA = 10, 20, "geman_mcclure", 0.3
WORKLOAD = ("cfg2: icp_odometry + grid_sample(0.3) preprocessing, synthetic 64x2048 rotating-LiDAR stream, "
            "kd-tree local map (20 frames), point-to-plane GN geman_mcclure 0.3, <=10 alignments, CV init")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def committed_traffic(name):
    """DRAM bytes per launch of a kernel family from the ncu capture committed under profiles/ (produced by
    tools/gpu_r2.sh traffic from the same sources; the file names the commit it was taken at)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        return d.get(name), d.get("commit")
    except Exception:
        return None, None


def committed_limiter():
    """What bounds the kd correspondence family, from the committed ncu --set full capture (profiles/r2_kd_limiter.json):
    issue-slot utilisation, instruction counts, stalls of the three kernels of a first ICP iteration."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_kd_limiter.json")))
        return {"verdict": d["verdict"], "source": d["source"],
                **{k: {"issue_active_pct": v["issue_active_pct"], "warp_instructions": v["warp_instructions"],
                       "long_scoreboard_stall_per_issue": v["long_scoreboard_stall_per_issue"]} for k, v in d["kernels"].items()}}
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (rank 0 only)."""

    def __init__(self, index=0, enabled=True):
        self.index, self.rows, self._p, self._t, self.enabled = index, [], None, None, enabled

    def start(self):
        if not self.enabled:
            return
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self._p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                        "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self._p = None
            return
        self._t = threading.Thread(target=self._read, daemon=True)
        self._t.start()

    def _read(self):
        for line in self._p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.enabled:
            return None
        if self._p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self._p.terminate()
        try:
            self._p.wait(timeout=2)
        except Exception:
            self._p.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
                for nme, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(smax)) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def make_scans(n_frames, h=H, w=W):
    from pylidar_slam_b200 import synthetic as syn
    return [syn.scan(k, h, w) for k in range(n_frames)]


def ref_vs_port_note():
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ref_vs_port.json")))
        return (f"; in the build container ({d['cores']} cores) the unmodified reference runs this stream at "
                f"{d['reference_ms_per_frame']:.0f} ms/frame and this port at {d['port_ms_per_frame']:.0f} ms/frame "
                f"(profiles/ref_vs_port.json)")
    except Exception:
        return ""


# ------------------------------------------------------------------------------------------ CPU arm
def run_cpu_port(scans, warmup, steps, threads=None, calibrate=False):
    """The oracle port of the reference path on the host cores; returns (fps, ms/frame list, calibration dict, last pose).

    calibrate=True gives the CPU arm the thread counts that are FASTEST on this host, not simply all of them: the path is
    made of many small tensor ops and short kd-tree queries, and 64 intra-op threads were measured slower than one on the
    64-core B200 hosts (SCALE_r01: 297 vs 369 ms/frame).  After the warm-up frames every candidate replays the SAME next two
    frames on a deep copy of the algorithm's state (local map, kd-tree, poses), twice; first the torch intra-op thread
    count (kd queries on all cores), then the worker count of scipy's cKDTree queries (pykdtree, which the reference uses,
    is OpenMP-parallel); the fastest pair runs the timed frames."""
    import copy
    import torch
    from oracle import icp_oracle as orc
    if threads:
        torch.set_num_threads(threads)
    cfg = orc.ICPConfig(max_num_alignments=MAX_ALIGN, data_key="input_data", local_map="kdtree", local_map_size=LM_SIZE,
                        scheme=SCHEME, sigma=SIGMA)
    algo = orc.ICPFrameToModelOracle(cfg, orc.Projector(H, W))
    kd_default = orc._KD_WORKERS

    def frame(a, k, prev):
        t0 = time.perf_counter()
        s, _ = orc.grid_sample(scans[k], VOXEL)                       # GridSample.filter
        dd = {"input_data": torch.from_numpy(s), "init_rpose": prev}  # ToTensor
        a.process_next_frame(dd)
        dt = time.perf_counter() - t0
        return dt, (dd["odometry_pose"].astype(np.float64) if "odometry_pose" in dd else prev)

    def fastest(cands, apply, k, prev):
        tried = {}
        for c in cands + cands[::-1]:                       # two rounds in opposite orders, the better one counts
            apply(c)
            a, p, dts = copy.deepcopy(algo), prev, []
            for j in range(k, min(k + 2, len(scans))):
                dt, p = frame(a, j, p)
                dts.append(dt)
            tried[c] = min(tried.get(c, 1e30), 1e3 * float(np.mean(dts)))
        best = min(tried, key=tried.get)
        apply(best)
        return best, tried

    def set_kd_workers(w):
        orc._KD_WORKERS = w

    prev, times, cal = None, [], {}
    try:
        for k in range(warmup + steps):
            if k == warmup and calibrate:
                ncpu = os.cpu_count() or 1
                cands = sorted({t for t in (1, 4, 8, 16, 32, ncpu) if t <= ncpu})
                _, cal["torch_tried_ms"] = fastest(cands, torch.set_num_threads, k, prev)
                kd_cands = sorted({w for w in (1, 8, 32) if w < ncpu}) + [-1]       # -1: all cores
                cal["kd_workers"], cal["kd_tried_ms"] = fastest(kd_cands, set_kd_workers, k, prev)
            dt, prev = frame(algo, k, prev)
            if k >= warmup:
                times.append(dt)
        cal["torch_threads"] = torch.get_num_threads()
        cal.setdefault("kd_workers", orc._KD_WORKERS)
    finally:
        orc._KD_WORKERS = kd_default
    return len(times) / sum(times), times, cal, prev


def threads_note(cal):
    if "torch_tried_ms" not in cal:
        return ""
    fmt = lambda d: ", ".join(f"{'all' if t == -1 else t}: {ms:.0f}" for t, ms in d.items())   # noqa: E731
    return ("; thread counts calibrated after the warm-up on copies of the state (best of two rounds of two frames, ms/frame) -- "
            f"torch intra-op threads {{{fmt(cal['torch_tried_ms'])}}} -> {cal['torch_threads']}, then cKDTree workers "
            f"{{{fmt(cal['kd_tried_ms'])}}} -> {'all' if cal['kd_workers'] == -1 else cal['kd_workers']}; host cores {os.cpu_count()}")


def reference_arm(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the map needs ~20 frames to reach steady state; more warm-up only costs CPU time
    warmup = min(args.warmup, 24)
    steps = args.steps
    scans = make_scans(warmup + steps)
    t0 = time.perf_counter()
    fps, times, cal, last_pose = run_cpu_port(scans, warmup, steps, calibrate=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"odometry_pose": np.asarray(last_pose, np.float64)})
    line = {
        "impl": "reference", "metric": "icp_odometry_frames_per_sec", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * float(np.mean(times)),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "height": H, "width": W, "voxel": VOXEL},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": os.cpu_count(), "torch_threads": cal["torch_threads"],
                         "kd_workers": cal["kd_workers"], "kind": "port",
                         "sample": f"frames {warmup}..{warmup + steps - 1} of the same seeded stream after {warmup} warm-up "
                                   f"frames (oracle/icp_oracle.py: torch CPU + scipy cKDTree), "
                                   f"{time.perf_counter() - t0:.1f} s wall" + threads_note(cal) + ref_vs_port_note()},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ GPU arm
def pose_errors(Ta, Tb):
    Ta, Tb = np.asarray(Ta, np.float64), np.asarray(Tb, np.float64)
    dt = np.linalg.norm(Ta[:3, 3] - Tb[:3, 3]) / max(np.linalg.norm(Tb[:3, 3]), 1e-12)
    dR = Tb[:3, :3].T @ Ta[:3, :3]
    ang = np.linalg.norm(0.5 * np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]]))
    return float(dt), float(ang)


def b200_arm(args):
    import torch
    import torch.distributed as dist
    import pylidar_slam_b200 as b200
    from pylidar_slam_b200 import _lib
    from pylidar_slam_b200 import synthetic as syn

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cpus = None
    if world > 1:
        # one process per GPU on a two-socket host: every rank stays on its GPU's socket (launches, pinned buffers and the
        # GPU's writes into mapped host memory do not cross the inter-socket link); a no-op wherever it cannot apply
        from pylidar_slam_b200.distributed import pin_to_gpu_numa
        numa_cpus = pin_to_gpu_numa(local_rank)
        dist.init_process_group("nccl", device_id=dev)

    W_, K_ = args.warmup, args.steps
    n_frames = 1 + W_ + K_
    scans = make_scans(n_frames)
    n_raw = scans[0].shape[0]
    stream = torch.cuda.Stream(device=dev)
    peak, peak_src = measured_peaks()

    comm_used = [args.comm]  # init_comm reports a fall-back from p2p to nccl

    def connect(ctx):
        if world > 1:
            from pylidar_slam_b200.distributed import init_comm
            comm_used[0] = init_comm(ctx, dist, rank, world, dev, mode=args.comm)

    def make_algo(local_map="kdtree", h=H, w=W, data_key="input_data", max_align=MAX_ALIGN, threshold=1e-4, comm=True):
        projector = b200.SphericalProjector(height=h, width=w, up_fov=3.0, down_fov=-24.0)
        lm = b200.KdTreeLocalMapConfig(local_map_size=LM_SIZE) if local_map == "kdtree" else \
            b200.ProjectiveLocalMapConfig(local_map_size=LM_SIZE)
        cfg = b200.ICPFrameToModelConfig(
            local_map=lm, alignment=b200.GaussNewtonPointToPlaneConfig(gauss_newton_config=dict(scheme=SCHEME, sigma=SIGMA, max_iters=1)),
            max_num_alignments=max_align, threshold_delta_pose=threshold, data_key=data_key)
        algo = b200.ICPFrameToModel(cfg, projector=projector, device=dev, stream=stream.cuda_stream)
        algo.init()
        if comm:
            connect(algo.ctx)
        return algo

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def flush_l2():
        with torch.cuda.stream(stream):
            flush_buf.zero_()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def hold_clocks(ms=80.0):
        """Keeps the GPU busy (L2-flush memsets, no step of the workload) right before a timed bracket: with the
        driver's short runs (5 warm-up frames = 3 ms of GPU work after seconds of host-side set-up) the SM clock is
        otherwise still ramping up inside the bracket."""
        t0 = time.perf_counter()
        while (time.perf_counter() - t0) * 1e3 < ms:
            for _ in range(8):
                flush_l2()
            torch.cuda.synchronize(dev)

    def max_over_ranks(*vals):
        if world == 1:
            return vals
        t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return tuple(float(v) for v in t.cpu())

    # ---------------- value: inputs resident in HBM, one C-ABI call per frame
    dev_scans = torch.from_numpy(np.stack(scans)).to(dev)
    torch.cuda.synchronize(dev)

    def device_pass(profile_slot=None, flush_each_step=False):
        """W warm-up frames, then exactly K timed frames inside ONE CUDA-event bracket on the library's
        stream (the local-map update of frame k runs on the library's second stream and overlaps frame
        k+1, so per-step brackets with untimed gaps would hide work; the bracket closes only after
        pls_synchronize has drained both streams)."""
        algo = make_algo()
        ctx = algo.ctx
        pose = np.zeros((4, 4), np.float32)
        params = np.zeros(6, np.float32)
        info = np.zeros(12, np.float64)
        has = C.c_int(0)
        prev = None
        launches0, iters, sharded = 0, [], 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for k in range(n_frames):
            timed = k > W_
            if k == W_ + 1:
                ctx.call("pls_synchronize")
                hold_clocks()
                flush_l2()
                barrier()
                launches0 = ctx.launch_count()
                if profile_slot is not None:
                    ctx.call("pls_profile_enable", profile_slot, 1)
                e0.record(stream)
            if timed and flush_each_step:
                flush_l2()        # inside the bracket: counted
            ctx.call("pls_process_frame_grid_sample", dev_scans[k].data_ptr(), n_raw, VOXEL, _lib.INPUT_TENSOR,
                     _lib.ptr(prev), _lib.ptr(pose), _lib.ptr(params), C.byref(has), _lib.ptr(info))
            if timed:
                iters.append(int(info[0]))
                sharded += int(info[11])
            if has.value:
                prev = pose.copy()
        ctx.call("pls_synchronize")
        e1.record(stream)
        barrier()
        launches = ctx.launch_count() - launches0
        total_ms = e0.elapsed_time(e1)
        prof = ctx.profile(profile_slot) if profile_slot is not None else None
        stats = {"samples": int(info[4]), "queries": int(info[2]), "map_points": int(info[3]), "iters_mean": float(np.mean(iters)),
                 "iters_total": int(np.sum(iters)), "frames_sharded": sharded}
        last = {"odometry_pose": pose.copy(), "odometry_params": params.copy(), "frame_info": info.copy()}
        return total_ms, launches, prof, stats, last

    clocks = ClockSampler(local_rank, enabled=(rank == 0))
    clocks.start()
    # `value` = the MEDIAN of REPEATS independent passes (fresh context, W warm-up frames, exactly K timed frames each):
    # with the driver's --steps 20 one bracket is a 10 ms sample; every pass is listed in config.repeats
    value_passes = [device_pass() for _ in range(1 if args.quick else REPEATS)]
    clock_info = clocks.stop()
    ms_dev, launches, _, stats, last = sorted(value_passes, key=lambda r: r[0])[len(value_passes) // 2]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    if args.quick:
        (ms_dev,) = max_over_ranks(ms_dev)
        if world > 1:
            dist.destroy_process_group()
        if rank == 0:
            print(json.dumps({"quick": True, "n_gpus": world, "comm": comm_used[0] if world > 1 else None,
                              "ms_per_step": ms_dev / K_, "gpu_launches": launches, **stats}))
        return
    ms_dev_flushed, _, _, _, _ = device_pass(flush_each_step=True)
    # roofline passes: same frames with CUDA events around one kernel family inside the library
    _, _, prof_nn, stats_nn, _ = device_pass(profile_slot=0)
    _, _, prof_idx, _, _ = device_pass(profile_slot=3)
    _, _, prof_gs, _, _ = device_pass(profile_slot=4)

    # ---------------- e2e: reference-shaped Python API from pinned host buffers
    pinned = [torch.from_numpy(s).pin_memory() for s in scans]
    host_scans = [p.numpy() for p in pinned]

    def e2e_pass():
        pre = b200.Preprocessing(b200.PreprocessingConfig(filters={
            "2": dict(filter_name="grid_sample", voxel_size=VOXEL, pointcloud_key="numpy_pc"),
            "3": dict(filter_name="to_tensor", keys=dict(sample_points="input_data"))}))
        algo = make_algo()
        gs_ctx = algo.ctx
        for f in pre.filters:
            if hasattr(f, "ctx"):
                f.ctx = gs_ctx
        prev, h2d, d2h = None, 0, 0
        t_start = 0.0
        for k in range(n_frames):
            timed = k > W_
            if k == W_ + 1:
                gs_ctx.call("pls_synchronize")
                hold_clocks()
                flush_l2()
                barrier()
                t_start = time.perf_counter()
            dd = {"numpy_pc": host_scans[k], "init_rpose": prev}
            pre.forward(dd)
            algo.process_next_frame(dd)
            if "odometry_pose" in dd:
                prev = dd["odometry_pose"].astype(np.float64)
            if timed:
                S = dd["sample_points"].shape[0]
                h2d += host_scans[k].nbytes + 64              # the raw scan + the initial pose (the samples stay on the device)
                d2h += S * 12 + S * 8 + 32 + 2176             # samples + indices (filter outputs) + count + FrameResult block
        gs_ctx.call("pls_synchronize")
        t = time.perf_counter() - t_start
        barrier()
        return t, h2d, d2h

    e2e_passes = [e2e_pass() for _ in range(REPEATS)]     # same rule as `value`: the median pass
    t_e, h2d, d2h = sorted(e2e_passes, key=lambda r: r[0])[len(e2e_passes) // 2]

    t_dev, t_e = max_over_ranks(ms_dev / 1e3, t_e)

    # ---------------- N > 1: sharded == single-GPU evidence on the benched stream (forced sharding, fixed iterations)
    # (the two sections below are evidence beside the headline: if one of them fails, the line above them is still printed)
    parity = None
    if world > 1:
        try:
            parity = sharded_vs_single(b200, make_algo, syn, dist, dev, rank, world, comm_used)
        except Exception as e:
            traceback.print_exc()
            parity = {"failed": f"{type(e).__name__}: {e}"}

    # ---------------- the HBM-sized configurations
    extra = None
    if not args.no_extra:
        try:
            extra = extra_workloads(b200, _lib, syn, make_algo, stream, dev, rank, world, dist, peak, comm_used, max_over_ranks,
                                    barrier)
        except Exception as e:
            traceback.print_exc()
            extra = {"failed": f"{type(e).__name__}: {e}"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    traffic, traffic_commit = committed_traffic("kd_iteration_bytes_per_launch")
    nn_ms, nn_launches, nn_bytes = prof_nn
    per_launch_bytes = nn_bytes / max(nn_launches, 1)
    avg_us = 1e3 * nn_ms / max(nn_launches, 1)
    achieved = per_launch_bytes / (avg_us * 1e-6) / 1e9 if nn_ms > 0 else 0.0
    lower = (stats_nn["queries"] * 44.0 + stats_nn["queries"] * 16.0) / (avg_us * 1e-6) / 1e9 if nn_ms > 0 else 0.0
    frame_ms = ms_dev / K_
    line = {
        "metric": "icp_odometry_frames_per_sec", "value": K_ / t_dev, "unit": "frames/s", "n_gpus": world,
        "steps": K_, "warmup": W_, "ms_per_step": 1e3 * t_dev / K_, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "height": H, "width": W, "voxel": VOXEL,
                   "clock_hold": "80 ms of L2-flush memsets (no workload step) right before each timed bracket, so that the "
                                 "SM clock is not still ramping up inside a 10 ms bracket",
                   "l2": "L2 flushed once before the timed bracket; every step streams a NEW 1.5 MB scan from HBM while the "
                         "~60 MB local map legitimately stays L2-resident across frames (production behaviour); "
                         "value_l2_flushed_every_step re-measures with a 256 MiB flush INSIDE the bracket before every frame",
                   "value_l2_flushed_every_step": K_ / (ms_dev_flushed / 1e3),
                   "repeats": {"rule": f"value and e2e are each the MEDIAN of {REPEATS} independent passes (fresh context, W warm-up "
                                       f"frames, exactly K timed frames in one bracket); at N > 1 the max over ranks of the ranks' "
                                       f"medians; the lists are rank 0's passes in run order",
                               "value_ms_per_step": [r[0] / K_ for r in value_passes],
                               "e2e_ms_per_step": [1e3 * r[0] / K_ for r in e2e_passes]},
                   "parallelism": "1 GPU" if world == 1 else
                   (f"{world} GPUs, map replicated; a frame's {stats['queries']} queries are below the sharding threshold "
                    f"(PLS_SHARD_MIN = 24576 per rank), so every rank runs the whole frame and no exchange takes place "
                    f"(frames sharded in the timed region: {stats['frames_sharded']}); the sharded path is measured on the "
                    f"HBM-sized configurations under extra_workloads ({comm_used[0]} exchange)"),
                   "host_cpus_rank0": numa_cpus if numa_cpus else "not pinned",
                   **{k: v for k, v in stats.items() if k != "iters_total"}},
        "e2e": {"value": K_ / t_e, "unit": "frames/s", "h2d_bytes_per_step": int(h2d / K_), "d2h_bytes_per_step": int(d2h / K_),
                "ms_per_step": 1e3 * t_e / K_},
        "gpu_launches": int(launches),
        "clocks": clock_info,
        "roofline": {"bound": "hbm", "kernel": "kd_nn_verify_kernel + kd_nn_warp_kernel + kd_normals_warp_kernel + kd_residual_kernel: "
                               "one executed ICP iteration (exact 1-NN, lazy 10-NN normals, point-to-plane reduction + fused solve)",
                     "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                     "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source":
                     f"profiles/r2_traffic.json (ncu dram bytes of the same kernels, commit {traffic_commit})" if traffic else None,
                     "launches": int(nn_launches), "avg_us": avg_us,
                     "algorithmic_bytes_per_launch": per_launch_bytes,
                     "algorithmic_bytes_formula": "SURVEY 8d: per query 12 + 27*8 + 4 B, 16 B per 1-NN candidate tested; per computed "
                                                  "normal 32 B + 16 B per k-NN candidate tested; 36 B per correspondence + 240 B per "
                                                  "block (candidates counted by the kernels)",
                     "lower_bound": {"achieved": lower, "frac": lower / peak if peak else None,
                                     "note": "44 B per query + 16 B per touched map point: the ~60 MB map is L2-resident, so this "
                                             "latency-bound family cannot approach the HBM roofline at 32 k queries per frame"},
                     "limiter": committed_limiter(),
                     "share_of_step": (nn_ms / K_) / frame_ms},
        "kernels": {"index_build_ms_per_frame": prof_idx[0] / K_, "grid_sample_ms_per_frame": prof_gs[0] / K_,
                    "correspondence_ms_per_frame": nn_ms / K_},
    }
    if parity is not None:
        line["config"]["sharded_vs_single"] = parity
    if extra is not None:
        line["config"]["extra_workloads"] = extra
    if world == 1 and not args.no_cpu:
        t0 = time.perf_counter()
        nb = min(len(scans), 30)
        fps_cpu, times, cal, _ = run_cpu_port(scans[:nb], min(22, nb - 6), nb - min(22, nb - 6), calibrate=True)
        line["cpu_baseline"] = {"value": fps_cpu, "unit": "frames/s", "cores": os.cpu_count(), "torch_threads": cal["torch_threads"],
                                "kd_workers": cal["kd_workers"], "kind": "port",
                                "sample": f"frames {min(22, nb - 6)}..{nb - 1} of the same stream (oracle port: torch CPU + scipy "
                                          f"cKDTree), {time.perf_counter() - t0:.1f} s wall" + threads_note(cal) + ref_vs_port_note()}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def sharded_vs_single(b200, make_algo, syn, dist, dev, rank, world, comm_used):
    """The sharded odometry (PLS_SHARD_MIN forced to 1: the 32 k queries of a frame split over the ranks, one exchange
    per ICP iteration) against rank 0's private single-GPU context on the first frames of the benched stream, with a
    fixed iteration count so that the stop rule cannot flip."""
    import torch
    frames = 8

    def drive(algo):
        prev, poses = None, []
        for k in range(frames):
            s, _ = b200.grid_sample(syn.scan(k, H, W), VOXEL, ctx=algo.ctx)
            dd = {"input_data": torch.from_numpy(s), "init_rpose": prev}
            algo.process_next_frame(dd)
            if "odometry_pose" in dd:
                prev = dd["odometry_pose"].astype(np.float64)
                poses.append(prev)
        return np.stack(poses), int(algo.last_info[11])

    from pylidar_slam_b200 import _lib
    _lib.load().pls_set_shard_min(1)
    sharded, was_sharded = drive(make_algo(max_align=6, threshold=0.0))
    _lib.load().pls_set_shard_min(-1)
    gathered = [torch.zeros_like(torch.from_numpy(sharded)).to(dev) for _ in range(world)]
    dist.all_gather(gathered, torch.from_numpy(sharded).to(dev))
    out = None
    if rank == 0:
        single, _ = drive(make_algo(max_align=6, threshold=0.0, comm=False))
        identical = all(bool((g.cpu().numpy() == sharded).all()) for g in gathered)
        errs = [pose_errors(a, b) for a, b in zip(sharded, single)]
        out = {"frames": frames - 1, "iterations_per_frame": 6, "exchange": comm_used[0], "sharded": bool(was_sharded),
               "max_rel_dt": max(e[0] for e in errs), "max_dR": max(e[1] for e in errs), "identical_across_ranks": identical}
    return out


def extra_workloads(b200, _lib, syn, make_algo, stream, dev, rank, world, dist, peak, comm_used, max_over_ranks, barrier):
    """cfg3 / cfg5 (projective map, the HBM-bound correspondence kernel) and cfg4 (5 M-point kd map).  At N > 1 the
    correspondences are sharded over the ranks (tiles / queries) with one 30-double exchange per ICP iteration."""
    import torch
    out = {}

    def timed_frames(algo, frames, warm, slot, feed):
        ctx = algo.ctx
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        prev, iters, sharded = None, 0, 0
        for k, data in enumerate(frames):
            if k == warm:
                ctx.call("pls_synchronize")
                barrier()
                ctx.call("pls_profile_enable", slot, 1)
                e0.record(stream)
            dd = feed(data)
            dd["init_rpose"] = prev
            algo.process_next_frame(dd)
            if "odometry_pose" in dd:
                prev = dd["odometry_pose"].astype(np.float64)
            if k >= warm:
                iters += int(algo.last_info[0])
                sharded += int(algo.last_info[11])
        ctx.call("pls_synchronize")
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        kms, klaunches, kbytes = ctx.profile(slot)
        n = len(frames) - warm
        (ms,) = max_over_ranks(ms)
        return ms / n, iters / n, kms, klaunches, kbytes, sharded

    # ---- projective configurations: one vertex map per frame, device-resident
    for name, (h, w, max_align, threshold, timed) in {"cfg3": (128, 2048, 10, 1e-4, 8), "cfg5": (128, 4096, 20, 0.0, 5)}.items():
        warm = 22
        vms = [torch.from_numpy(syn.vertex_map_from_scan(syn.scan(k, h, w), h, w)).to(dev) for k in range(warm + timed)]
        algo = make_algo(local_map="projective", h=h, w=w, data_key="vertex_map", max_align=max_align, threshold=threshold)
        ms_frame, iters, kms, kl, kb, sharded = timed_frames(algo, vms, warm, 1, lambda vm: {"vertex_map": vm})
        traffic, tcommit = committed_traffic(f"{name}_proj_bytes_per_launch")
        us = 1e3 * kms / max(kl, 1)
        ach = (kb / max(kl, 1)) / (us * 1e-6) / 1e9 if kms > 0 else 0.0
        out[name] = {"workload": f"{h}x{w} vertex maps, projective local map (20 frames), {max_align} alignments"
                                 + (" (all executed: threshold_delta_pose = 0)" if threshold == 0.0 else " at most"),
                     "ms_per_frame": ms_frame, "frames_per_sec": 1e3 / ms_frame, "iterations_per_frame": iters, "timed_frames": timed,
                     "kernel": "proj_icp_tma_kernel", "kernel_avg_us": us, "kernel_launches": int(kl),
                     "algorithmic_bytes_per_launch": kb / max(kl, 1), "achieved_gbs": ach, "frac_of_measured_hbm_peak": ach / peak,
                     "traffic_bytes_per_launch": traffic, "traffic_commit": tcommit,
                     "ranks": world, "tiles_sharded": bool(sharded), "exchange": comm_used[0] if world > 1 else None,
                     "kernel_note": "per rank: each rank streams its share of the tiles" if world > 1 else None}
        del algo, vms
        torch.cuda.empty_cache()

    # ---- cfg4: 5 M-point kd map, one 64x2048 scan registered against it (fixed 5 iterations)
    target = 5_000_000
    frames_needed = (target + H * W - 1) // (H * W)
    world_pts = []
    for k in range(frames_needed):
        P = syn.gt_pose(100 + 3 * k)
        pc = syn.scan(100 + 3 * k, H, W).astype(np.float64)
        world_pts.append((pc @ P[:3, :3].T + P[:3, 3]).astype(np.float32))
    cloud = np.concatenate(world_pts)[:target]
    algo = make_algo(max_align=5, threshold=0.0, data_key="numpy_pc")
    ctx = algo.ctx
    cloud_dev = torch.from_numpy(cloud).to(dev)
    eye = np.eye(4, dtype=np.float32)
    ctx.call("pls_kdmap_update_points", _lib.ptr(eye), cloud_dev.data_ptr(), cloud.shape[0])
    Pq = syn.gt_pose(100 + 3 * (frames_needed // 2))
    q = ((syn.scan(100 + 3 * (frames_needed // 2), H, W).astype(np.float64) + np.array([0.05, -0.03, 0.01])) @ Pq[:3, :3].T
         + Pq[:3, 3]).astype(np.float32)
    q_dev = torch.from_numpy(q).to(dev)
    T, params, losses, it = np.zeros((4, 4), np.float32), np.zeros(6, np.float32), np.zeros(5, np.float32), C.c_int(0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps, ms_reg = 4, []
    for r in range(reps + 1):
        if r == 1:
            ctx.call("pls_profile_enable", 0, 1)
        barrier()
        e0.record(stream)
        ctx.call("pls_register_frame", q_dev.data_ptr(), q.shape[0], None, _lib.ptr(T), _lib.ptr(params), _lib.ptr(losses), C.byref(it))
        e1.record(stream)
        torch.cuda.synchronize(dev)
        if r >= 1:
            ms_reg.append(e0.elapsed_time(e1))
    kms, kl, kb = ctx.profile(0)
    (ms4,) = max_over_ranks(float(np.mean(ms_reg)))
    us = 1e3 * kms / max(kl, 1)
    ach = (kb / max(kl, 1)) / (us * 1e-6) / 1e9 if kms > 0 else 0.0
    out["cfg4"] = {"workload": f"{cloud.shape[0]} map points (kd map), one 64x2048 scan ({q.shape[0]} queries) registered with 5 ICP "
                               f"iterations (threshold_delta_pose = 0)",
                   "ms_per_registration": ms4, "iterations": int(it.value), "kernel": "kd correspondence family (per executed iteration)",
                   "kernel_avg_us": us, "kernel_launches": int(kl), "algorithmic_bytes_per_launch": kb / max(kl, 1),
                   "achieved_gbs": ach, "frac_of_measured_hbm_peak": ach / peak, "ranks": world,
                   "queries_sharded": bool(ctx_sharded(ctx)), "exchange": comm_used[0] if world > 1 else None}
    return out


def ctx_sharded(ctx):
    n = C.c_int(0)
    ctx.lib.pls_last_sharded(ctx.handle, C.byref(n))
    return n.value


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=24)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip config.extra_workloads (cfg3 / cfg4 / cfg5)")
    ap.add_argument("--quick", action="store_true", help="device-resident pass only (for ncu captures)")
    ap.add_argument("--comm", default="p2p", choices=["p2p", "nccl"],
                    help="N>1 exchange: one-shot NVLink peer-to-peer all-reduce fused into the solve kernel, or NCCL")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed path's outputs of its last timed frame to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
