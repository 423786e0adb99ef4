"""bench.py's CPU arm (the oracle port timed on the host cores): the thread calibration replays frames on COPIES of the
algorithm's state and must leave the timed stream untouched; the --impl reference line keeps the contract's keys."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_thread_calibration_does_not_disturb_the_stream(monkeypatch):
    import torch
    import bench
    from oracle import icp_oracle as orc
    before = torch.get_num_threads()
    try:
        scans = bench.make_scans(5)
        _, t_plain, cal_plain, pose_plain = bench.run_cpu_port(scans, 2, 3, threads=1)
        assert "torch_tried_ms" not in cal_plain and cal_plain["torch_threads"] == 1 and cal_plain["kd_workers"] == -1
        # one torch candidate (a "single-core host"): the calibration replays two frames on deep copies of the state, and
        # the timed frames then run with the same torch thread count as the plain run (kd queries are exact whatever the
        # worker count) -- the arithmetic must be IDENTICAL
        monkeypatch.setattr(bench.os, "cpu_count", lambda: 1)
        _, t_cal, cal, pose_cal = bench.run_cpu_port(scans, 2, 3, threads=1, calibrate=True)
        assert len(t_plain) == len(t_cal) == 3
        assert cal["torch_threads"] == 1 and list(cal["torch_tried_ms"]) == [1] and list(cal["kd_tried_ms"]) == [-1]
        np.testing.assert_array_equal(pose_cal, pose_plain)
        monkeypatch.undo()
        # several candidates: every one is tried, the fastest is kept, the oracle's default is restored afterwards
        n = os.cpu_count()
        _, _, cal, pose_multi = bench.run_cpu_port(scans, 2, 2, calibrate=True)
        assert set(cal["torch_tried_ms"]) == {t for t in (1, 4, 8, 16, 32, n) if t <= n}
        assert set(cal["kd_tried_ms"]) == {w for w in (1, 8, 32) if w < n} | {-1}
        assert cal["torch_threads"] == min(cal["torch_tried_ms"], key=cal["torch_tried_ms"].get) == torch.get_num_threads()
        assert cal["kd_workers"] == min(cal["kd_tried_ms"], key=cal["kd_tried_ms"].get) and orc._KD_WORKERS == -1
        assert "cKDTree workers" in bench.threads_note(cal)
        np.testing.assert_allclose(pose_multi[:3, 3], pose_plain[:3, 3], rtol=0, atol=0.2)   # (another frame: same motion model)
    finally:
        torch.set_num_threads(before)


def test_reference_arm_prints_one_contract_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3",
                          "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env={**os.environ, "RANK": "0"})
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "icp_odometry_frames_per_sec" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 3 and d["gpu_launches"] == 0
    assert d["value"] > 0 and abs(d["value"] - 1e3 / d["ms_per_step"]) / d["value"] < 1e-6
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] == os.cpu_count() and cb["torch_threads"] >= 1
    assert cb["kd_workers"] in (-1, 1, 8, 32) and "calibrated" in cb["sample"]
    assert d["config"]["workload"].startswith("cfg2") and d["config"]["height"] == 64 and d["config"]["width"] == 2048
    assert os.listdir(tmp_path) == ["odometry_pose.npy"]
    pose = np.load(tmp_path / "odometry_pose.npy")
    assert pose.shape == (4, 4) and pose.dtype == np.float64 and np.isfinite(pose).all()


def test_reference_arm_is_silent_on_other_ranks():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env={**os.environ, "RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0 and out.stdout.strip() == ""


# ------------------------------------------------------------------------------------------------------------------
# The GPU arm's CONTROL FLOW without a GPU: bench.b200_arm runs against a test-only stand-in for the C ABI (the oracle
# behind tests/dryrun_next_rows.FakeContext) and stand-ins for the few torch.cuda objects it touches.  This checks that
# the bench line is assembled (keys, the median-of-passes rule, byte counts) -- never a number: the timings below are CPU
# times of the oracle and mean nothing.  The product has no such path; the stand-ins live in this file only.
def _bench_fakes(monkeypatch):
    import contextlib
    import time
    import ctypes as C
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import dryrun_next_rows as dry
    from oracle import icp_oracle as orc
    from pylidar_slam_b200 import _lib, common

    class BenchFakeContext(dry.FakeContext):
        launches = 0

        def __init__(self, **kwargs):
            kwargs.pop("stream", None)
            super().__init__(**kwargs)
            self.handle, self.lib = None, None

        def pls_synchronize(self):
            pass

        def pls_comm_p2p_handle(self, world, buf):          # distributed.init_comm's rendezvous (p2p mode)
            for i in range(64):
                buf[i] = (i + 1) % 256

        def pls_comm_p2p_init(self, world, rank, raw):
            assert len(raw) == 64 * world

        def pls_profile_enable(self, slot, on):
            pass

        def launch_count(self):
            return BenchFakeContext.launches

        def profile(self, which, reset=True):
            return 1.0, 2, 1.0e6

        def pls_process_frame(self, *a):
            BenchFakeContext.launches += 30
            return super().pls_process_frame(*a)

        def pls_process_frame_grid_sample(self, raw, n, voxel, layout, init, pose, params, has, info):
            s, _ = orc.grid_sample(dry.arr(raw, (n, 3), np.float32), voxel)
            s = np.ascontiguousarray(s, dtype=np.float32)
            self.pls_process_frame(s.ctypes.data, layout, len(s), init, pose, params, has, info)
            dry.arr(info, (12,), np.float64)[4] = len(s)

    class FakeStream:
        def __init__(self, device=None):
            self.cuda_stream = 0

    class FakeEvent:
        def __init__(self, enable_timing=False):
            self.t = 0.0

        def record(self, stream=None):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return 1e3 * (other.t - self.t)

    real_empty, real_to = torch.empty, torch.Tensor.to

    def empty(*a, **k):
        if "device" in k and torch.device(k["device"]).type == "cuda":
            k["device"] = "cpu"
            a = (1 << 16,)                                      # the 256 MiB L2-flush buffer
        return real_empty(*a, **k)

    def on_cpu(fn):                                          # factory calls with device=cuda:* build CPU tensors here
        def wrapped(*a, **k):
            if "device" in k and k["device"] is not None and torch.device(k["device"]).type == "cuda":
                k["device"] = "cpu"
            return fn(*a, **k)
        return wrapped

    def to(self, *a, **k):
        if a and isinstance(a[0], torch.device) and a[0].type == "cuda":
            return self
        return real_to(self, *a, **k)

    monkeypatch.setattr(_lib, "Context", BenchFakeContext)
    monkeypatch.setattr(common, "_default_ctx", BenchFakeContext())
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(torch.cuda, "Stream", FakeStream)
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda d=None: None)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "empty_cache", lambda: None)
    monkeypatch.setattr(torch, "empty", empty)
    monkeypatch.setattr(torch, "tensor", on_cpu(torch.tensor))
    monkeypatch.setattr(torch, "zeros", on_cpu(torch.zeros))
    monkeypatch.setattr(torch.Tensor, "to", to)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self)
    return BenchFakeContext


def test_b200_arm_assembles_the_contract_line_dry_run(monkeypatch, capsys, tmp_path):
    import argparse
    import bench
    from pylidar_slam_b200 import _lib
    real_context = _lib.Context
    _bench_fakes(monkeypatch)
    monkeypatch.setattr(bench.ClockSampler, "start", lambda self: None)
    monkeypatch.setattr(bench.ClockSampler, "stop", lambda self: {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["dry run"]})
    from pylidar_slam_b200 import synthetic as syn
    monkeypatch.setattr(bench, "H", 32)        # a small sensor keeps the oracle-backed frames at a few tens of ms
    monkeypatch.setattr(bench, "W", 512)
    monkeypatch.setattr(bench, "VOXEL", 0.4)
    monkeypatch.setattr(bench, "make_scans", lambda n, h=32, w=512: [syn.scan(k, h, w) for k in range(n)])
    for k in ("WORLD_SIZE", "RANK", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    def failing_extras(*a, **k):                # an extra workload that dies must not take the headline line with it
        raise RuntimeError("extra workload failed (dry run)")
    monkeypatch.setattr(bench, "extra_workloads", failing_extras)
    args = argparse.Namespace(gpus=1, steps=4, warmup=3, impl="b200", no_cpu=False, no_extra=False, quick=False, comm="p2p",
                              dump_outputs=str(tmp_path / "out"))
    bench.b200_arm(args)
    lines = [l for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    # --dump-outputs: the last timed frame's outputs of the timed call (frame 1 + W + K - 1 of the seeded stream)
    dumped = {f: np.load(tmp_path / "out" / f) for f in sorted(os.listdir(tmp_path / "out"))}
    assert {f: (a.shape, a.dtype) for f, a in dumped.items()} == {
        "frame_info.npy": ((12,), np.float64), "odometry_params.npy": ((6,), np.float32), "odometry_pose.npy": ((4, 4), np.float32)}
    assert np.isfinite(dumped["odometry_pose.npy"]).all() and not np.array_equal(dumped["odometry_pose.npy"], np.eye(4))
    assert dumped["frame_info.npy"][0] >= 1 and dumped["frame_info.npy"][4] == d["config"]["samples"]
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "kernels"):
        assert key in d, key
    assert d["metric"] == "icp_odometry_frames_per_sec" and d["unit"] == "frames/s" and d["n_gpus"] == 1
    assert d["steps"] == 4 and d["warmup"] == 3 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert abs(d["value"] - 1e3 / d["ms_per_step"]) / d["value"] < 1e-9
    rep = d["config"]["repeats"]
    assert len(rep["value_ms_per_step"]) == bench.REPEATS and len(rep["e2e_ms_per_step"]) == bench.REPEATS
    assert abs(sorted(rep["value_ms_per_step"])[bench.REPEATS // 2] - d["ms_per_step"]) < 1e-9       # the median pass
    assert abs(sorted(rep["e2e_ms_per_step"])[bench.REPEATS // 2] - d["e2e"]["ms_per_step"]) < 1e-9
    assert d["e2e"]["unit"] == "frames/s" and abs(d["e2e"]["value"] - 1e3 / d["e2e"]["ms_per_step"]) / d["e2e"]["value"] < 1e-9
    assert d["e2e"]["h2d_bytes_per_step"] == 32 * 512 * 12 + 64 and d["e2e"]["d2h_bytes_per_step"] > 2176
    assert d["gpu_launches"] == 30 * 4                                                                 # launches of the timed frames only
    r = d["roofline"]
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert key in r, key
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert d["config"]["workload"].startswith("cfg2")
    cb = d["cpu_baseline"]                                                                             # the CPU leg at N = 1
    assert cb["kind"] == "port" and cb["unit"] == "frames/s" and cb["value"] > 0 and cb["cores"] == os.cpu_count()
    assert cb["torch_threads"] >= 1 and "calibrated" in cb["sample"]
    assert d["config"]["extra_workloads"] == {"failed": "RuntimeError: extra workload failed (dry run)"}
    assert _lib.Context is not real_context                                                            # still patched here ...


def test_bench_fakes_do_not_leak():
    from pylidar_slam_b200 import _lib
    assert _lib.Context.__name__ == "Context" and _lib.Context.__module__ == "pylidar_slam_b200._lib"   # ... and restored after


# ---- the same dry run on TWO ranks (gloo): max over ranks, the barriers inside the repeated passes, the parity section
class _Patch:
    """monkeypatch's setattr / delenv for a worker process (nothing to undo: the process exits)."""

    @staticmethod
    def setattr(obj, name, value):
        setattr(obj, name, value)

    @staticmethod
    def delenv(name, raising=False):
        os.environ.pop(name, None)


def _two_rank_worker(rank, world, port, out):
    import argparse
    import contextlib
    import io
    import torch
    import torch.distributed as dist
    import bench
    from pylidar_slam_b200 import synthetic as syn
    os.environ.update({"MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(port), "RANK": str(rank), "WORLD_SIZE": str(world),
                       "LOCAL_RANK": "0"})
    _bench_fakes(_Patch)
    real_init = dist.init_process_group
    dist.init_process_group = lambda backend, device_id=None: real_init("gloo", rank=rank, world_size=world)
    bench.ClockSampler.start = lambda self: None
    bench.ClockSampler.stop = lambda self: {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["dry run"]} if self.enabled else None
    bench.H, bench.W, bench.VOXEL = 32, 512, 0.4
    bench.make_scans = lambda n, h=32, w=512: [syn.scan(k, h, w) for k in range(n)]
    bench.extra_workloads = lambda *a, **k: {"stub": True}
    torch.set_num_threads(1)
    args = argparse.Namespace(gpus=world, steps=3, warmup=3, impl="b200", no_cpu=False, no_extra=False, quick=False, comm="p2p",
                              dump_outputs=None)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        bench.b200_arm(args)
    out[rank] = buf.getvalue()


def test_b200_arm_two_ranks_dry_run():
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = mp.Manager().dict()
    mp.spawn(_two_rank_worker, args=(2, port, out), nprocs=2, join=True)
    assert out[1].strip() == ""                                     # rank 0 alone prints
    lines = [l for l in out[0].splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["n_gpus"] == 2 and d["steps"] == 3 and d["warmup"] == 3 and "cpu_baseline" not in d   # CPU leg at N = 1 only
    assert "2 GPUs" in d["config"]["parallelism"] and d["config"]["extra_workloads"] == {"stub": True}
    assert d["config"]["host_cpus_rank0"] == "not pinned"                                   # no GPU here: nothing to pin to
    par = d["config"]["sharded_vs_single"]
    assert par["identical_across_ranks"] is True and par["max_rel_dt"] == 0.0 and par["max_dR"] == 0.0 and par["exchange"] == "p2p"
    rep = d["config"]["repeats"]
    assert len(rep["value_ms_per_step"]) == len(rep["e2e_ms_per_step"]) == 3
    # the headline is the max over ranks of the ranks' medians: never below rank 0's own median
    assert d["ms_per_step"] >= sorted(rep["value_ms_per_step"])[1] - 1e-9
    assert d["e2e"]["ms_per_step"] >= sorted(rep["e2e_ms_per_step"])[1] - 1e-9


def test_committed_evidence_files_feed_the_bench_line():
    """bench.py attaches committed ncu evidence to its line (DRAM traffic per launch, the limiter digest, the
    reference-vs-port timing) and silently reports None when a file is missing or malformed: pin the files and the keys."""
    import bench
    traffic, commit = bench.committed_traffic("kd_iteration_bytes_per_launch")
    assert traffic and traffic > 1e6 and commit
    for name in ("cfg3_proj_bytes_per_launch", "cfg5_proj_bytes_per_launch"):
        t, c = bench.committed_traffic(name)
        assert t and t > 1e7 and c == commit
    lim = bench.committed_limiter()
    assert lim and lim["verdict"] and lim["source"]
    kernels = [k for k in lim if k not in ("verdict", "source")]
    assert len(kernels) >= 3 and all(0 < lim[k]["issue_active_pct"] <= 100 and lim[k]["warp_instructions"] > 0 for k in kernels)
    note = bench.ref_vs_port_note()
    assert "unmodified reference" in note and "profiles/ref_vs_port.json" in note
    peak, src = bench.measured_peaks()
    assert 3000 < peak < 9000 and ("MEASURED_PEAKS" in src or "fallback" in src)
