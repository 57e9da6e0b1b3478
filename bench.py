#!/usr/bin/env python
"""bench.py -- throughput of one outer bundle-adjustment iteration of the direct-BA hot path.

    python bench.py --gpus 1 --steps K --warmup W            # our sm_100a backend
    python bench.py --impl reference --gpus 1 --steps K ...  # the reference's own CUDA kernels (oracle/_ref)
    python bench.py ... --dump-outputs DIR                   # + what the last timed step computed, as DIR/<name>.npy

A "step" is ONE outer iteration of DirectBA::BundleAdjustment (surfel activation + geometry optimisation +
pose optimisation of every keyframe, direct_ba_alternating.cc:345-717) on a seeded synthetic 640x480 scene,
restarted from the same perturbed state every step (device-to-device restore inside the timed region), so
every step does the same work.  Metric (BASELINE.json): surfel-keyframe residuals per second =
(depth residuals + descriptor residuals at the pose step's starting state) / step time.

Prints exactly one JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the CPU baseline's OpenMP threads stay on their cores (read when the OpenMP runtime initialises)
os.environ.setdefault("OMP_PROC_BIND", "close")
os.environ.setdefault("OMP_PLACES", "cores")

METRIC = "surfel_keyframe_residuals_per_second_per_BA_iteration"
UNIT = "residuals/s"
# --dump-outputs: at most this many surfels (a fixed, seeded sample of a larger map) -> 8 rows + flags + indices, 44 MB
DUMP_SURFELS = 1 << 20
DUMP_RESULT_FIELDS = ("iterations_done", "converged", "depth_residual_count", "descriptor_residual_count", "cost",
                      "pose_iterations_total", "surfels_deleted", "surfels_size", "surfels_created", "surfels_merged")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons sampled WHILE the timed region runs (B200_PROFILING.md clocks line): NVML polled from a
    thread every millisecond (a timed region can be a few tens of ms), nvidia-smi -lms as the fallback."""

    _REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []
        self.samples = []
        self.mask = 0
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def _poll(self):
        n, h = self._nvml, self._handle
        while not self._stop.is_set():
            try:
                self.samples.append(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
                self.mask |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            except Exception:
                break
            time.sleep(0.001)

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()
            return
        except Exception:
            self._nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}",
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self._nvml is not None:
            self._stop.set()
            self._thread.join(timeout=1.0)
            reasons = sorted(name for bit, name in self._REASONS.items() if self.mask & bit)
            return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                    "reasons": reasons, "samples": len(self.samples), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def workload_name(scene):
    """config.workload -- the same string in both arms (the driver compares the two lines' configs)."""
    c = scene.cfg
    return (f"{c.name}: {c.num_keyframes} keyframes x {scene.num_surfels} surfels, {c.width}x{c.height}, 1 outer alternating-BA "
            "iteration (activation + geometry + poses), depth + descriptor residuals")


def algorithmic_bytes(prof, kf_evals):
    """SURVEY.md 8(d): bytes_pose_pass = 12 n_pair + 10 n_inimg + 2 n_depthok + 12 n_assoc + 12 n_photo + 108 K."""
    return (12 * prof["n_pair"] + 10 * prof["n_inimg"] + 2 * prof["n_depthok"] + 12 * prof["n_assoc"]
            + 12 * prof["n_photo"] + 108 * kf_evals)


def cpu_port_baseline(scene, max_kf=20, max_surfels=200_000, repeats=3):
    """The CPU oracle port on a bounded slice of the workload (first keyframes / first surfels)."""
    import copy
    from oracle import cpu_oracle
    K = min(scene.cfg.num_keyframes, max_kf)
    n = min(scene.num_surfels, max_surfels)
    sub = copy.copy(scene)
    sub.cfg = copy.copy(scene.cfg)
    sub.cfg.num_keyframes = K
    sub.depth, sub.normals, sub.radius, sub.color = scene.depth[:K], scene.normals[:K], scene.radius[:K], scene.color[:K]
    sub.poses_init, sub.poses_true = scene.poses_init[:K], scene.poses_true[:K]
    sub.min_depth, sub.max_depth = scene.min_depth[:K], scene.max_depth[:K]
    sub.num_surfels = n
    # threads = what the OpenMP runtime would use, but never more than the CPUs this process may run on (a shared box hands a job
    # a couple of cores while OMP_NUM_THREADS / the core count say 64: the baseline would then time 64 threads taking turns)
    lib_ = cpu_oracle.lib()
    cores = max(1, min(int(lib_.orc_get_max_threads()), len(os.sched_getaffinity(0))))
    lib_.orc_set_num_threads(cores)
    times = []
    for _ in range(repeats):   # best of `repeats` (a shared host: single runs varied 3x in round 1); threads pinned via OMP_PROC_BIND
        orc = cpu_oracle.Oracle(sub)
        t0 = time.perf_counter()
        r = orc.bundle_adjust(True, True, 1, 1)
        times.append(time.perf_counter() - t0)
    dt = min(times)
    residuals = r.n_assoc + 2 * r.n_photo
    return {"value": residuals / dt, "unit": UNIT, "cores": int(cores), "kind": "port",
            "sample": f"cfg2-sized slice of the workload: 1 outer BA iteration of oracle/badba_oracle.c (OpenMP, threads pinned) on the "
                      f"first {K} keyframes x first {n} surfels; best of {repeats} runs ({', '.join(f'{t:.2f}' for t in times)} s)"}


def run_ours(args, scene, rank, world):
    import torch
    from badslam_b200.direct_ba import DirectBA
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    K = scene.cfg.num_keyframes
    import torch.distributed as dist
    if world > 1:
        # one process per GPU (torchrun); keyframe images + surfels replicated, surfel shards / keyframe work list split
        if not dist.is_initialized():
            dist.init_process_group(backend="nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[dev.index])

    ba = DirectBA.from_scene(scene, device=dev, rank=rank, world_size=world)
    exchange = "none"
    if world > 1:
        ba.SetCollective()
        exchange = "nccl all-gather"
        if not os.environ.get("BADBA_NO_PEER"):
            try:   # geometry exchange fused into the kernels: stores into the peers' replicas over NVLink (CUDA IPC)
                if ba.EnablePeerExchange() == world - 1:
                    exchange = "nvlink peer stores from the geometry kernels + 1-element all-reduce barrier"
            except Exception as e:   # noqa: BLE001  (IPC not permitted in this environment: keep the NCCL exchange)
                exchange = f"nccl all-gather (peer mapping unavailable: {type(e).__name__})"
    surf = ba.surfels()
    backup = surf[:8].clone()
    poses0 = scene.poses_init.copy()
    act0 = np.zeros(K, np.int32)
    # A step = ONE iteration of the alternation on the full configured workload.  The end-of-scheme surfel maintenance
    # (PerformBASchemeEndTasks: delete / radius update / compaction) runs once per BundleAdjustment call, not per
    # iteration, and would change the surfel set between steps: it is kept out of the steps (increase_ba_iteration_count =
    # false with the counters in sync, direct_ba_alternating.cc:313-319) and is part of the full-BA number below.
    ba.SetLastBAIterationCount(ba.ba_iteration_count())

    # --intrinsics (cfg4): the depth-intrinsics / depth-deformation and colour-intrinsics steps are part of the iteration; the
    # camera model is restored before every step like the surfels and poses are.
    intr = bool(getattr(args, "intrinsics", False))
    if intr:
        cam0 = (ba.depth_camera(), ba.color_camera(), ba.a(), ba.cfactor_buffer().copy())

    def step():
        surf[:8].copy_(backup, non_blocking=True)
        if world > 1:
            ba.MarkReplicaRewritten()   # (the other ranks' geometry kernels store into this replica: fence them behind the restore)
        ba.SetKeyframeStates(poses0, act0)
        if intr:
            ba.SetDepthCamera(cam0[0]); ba.SetColorCamera(cam0[1]); ba.SetA(cam0[2]); ba.SetCFactorBuffer(cam0[3])
        return ba.BundleAdjustment(None, intr, intr, False, True, True, 1, 1, increase_ba_iteration_count=False)

    for _ in range(args.warmup):
        res = step()
    residuals = res.depth_residual_count + res.descriptor_residual_count
    torch.cuda.synchronize()
    ba.SetProfiling(2)          # one untimed step with the byte-model counters on: identical counts every step
    ba.GetProfile(reset=True)
    step()
    counts = ba.GetProfile(reset=True)
    ba.SetProfiling(1)          # the timed region only records cudaEvents around every pose-kernel launch
    launches0 = ba.kernel_launch_count()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize()
    ev0.record()
    stage = np.zeros(3)
    for _ in range(args.steps):
        res = step()
        stage += [res.ms_surfel_activation, res.ms_geometry_optimization, res.ms_pose_optimization]
    ev1.record()
    torch.cuda.synchronize()
    barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms_total = ev0.elapsed_time(ev1)
    if world > 1:   # device time, max over ranks
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    launches = ba.kernel_launch_count() - launches0
    prof = ba.GetProfile(reset=True)
    ba.SetProfiling(0)
    for key in ("n_pair", "n_inimg", "n_depthok", "n_assoc", "n_photo", "kf_evals"):
        prof[key] = counts[key] * args.steps
    value = residuals / (ms_step * 1e-3)

    # roofline of the dominant kernel (PoseAccumulateKernel), measured live with cudaEvents around each launch
    peak, peak_src = load_peaks()
    alg = algorithmic_bytes(prof, prof["kf_evals"])
    pose_s = prof["pose_ms"] * 1e-3
    achieved = alg / pose_s / 1e9 if pose_s > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "pose_kernel_dram_bytes_per_launch.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f).get(scene.cfg.name)
    roofline = {"bound": "hbm", "kernel": "PoseAccumulateKernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg / max(prof["pose_launches"], 1),
                "avg_launch_ms": prof["pose_ms"] / max(prof["pose_launches"], 1),
                "launches_timed": prof["pose_launches"],
                "kernel_share_of_step": prof["pose_ms"] / ms_total,
                "pairs_per_s": prof["n_pair"] / pose_s if pose_s > 0 else 0.0}

    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ba, res)

    multi_gpu_check = None
    if world > 1:
        multi_gpu_check = check_replicas(scene, ba, step, dev, rank, world)

    # full BA (10 continuing iterations) for the second headline number
    surf[:8].copy_(backup)
    if world > 1:
        ba.MarkReplicaRewritten()
    ba.SetKeyframeStates(poses0, act0)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    full = ba.BundleAdjustment(None, False, False, False, True, True, 10, 10)
    torch.cuda.synchronize()
    ms_full = (time.perf_counter() - t0) * 1e3
    del ba, surf, backup
    torch.cuda.empty_cache()

    # e2e: same step through the public API with HOST buffers: one keyframe's RGB-D images (pinned) + all poses go
    # host->device, poses/statistics come back, every step.
    e2e_all = None
    if world == 1:
        e2e = run_e2e(args, scene, dev, residuals)
        if not args.no_e2e_all:
            e2e_all = run_e2e(args, scene, dev, residuals, all_keyframes=True)
    else:
        e2e = run_e2e_multi(args, scene, dev, residuals, rank, world)

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(scene), "keyframes": K, "surfels": scene.num_surfels, "residuals_per_step": int(residuals),
                   "l2": "inputs larger than L2 (keyframe images + surfels)", "parallelism": f"gpus={world}"},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "stage_ms": {"BA_surfel_activation+normals": stage[0] / args.steps, "BA_geometry_optimization(position+descriptor)": stage[1] / args.steps,
                     "BA_pose_optimization": stage[2] / args.steps},
        "pose_iterations_per_step": res.pose_iterations_total,
        "ms_full_ba_10_iterations": ms_full, "full_ba_iterations": full.iterations_done,
    }
    if e2e_all is not None:
        out["e2e_all_keyframes"] = e2e_all
    if multi_gpu_check is not None:
        out["multi_gpu_check"] = multi_gpu_check
    # host side of the box (the Gauss-Newton loop of the pose step polls from a host thread per rank: a box whose cores are
    # oversubscribed by other tenants shows up here)
    out["host"] = {"cpus_available": len(os.sched_getaffinity(0)), "loadavg_1min": round(os.getloadavg()[0], 1)}
    if intr:
        out["config"]["intrinsics"] = "depth intrinsics + depth deformation + colour intrinsics optimised in every step (--intrinsics)"
        out["stage_ms"]["BA_intrinsics_optimization"] = res.ms_intrinsics_optimization
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_port_baseline(scene)
    if world > 1:
        out["config"]["parallelism"] = (f"gpus={world}: keyframe images + surfels replicated; geometry step sharded by 256-surfel "
                                        f"granules dealt round-robin (exchange: {exchange}), pose step sharded by keyframe, "
                                        "balanced by measured work (1 all-reduce of K x 17 floats); NCCL over NVLink")
        dist.barrier(device_ids=[dev.index])
    return out


def dump_outputs(out_dir, ba, res):
    """What the last timed step handed back to a caller, as float32 / float64 arrays in out_dir: keyframe poses and
    activations, the BundleAdjustment result counters (DUMP_RESULT_FIELDS) and the surfel rows 0-7 (bit patterns of the packed
    rows kept) with the active flags, of every surfel or of a fixed, seeded sample of DUMP_SURFELS of them."""
    os.makedirs(out_dir, exist_ok=True)
    poses, act = ba.GetKeyframeStates()
    rows, flags = ba.GetSurfelsHost(), ba.GetActiveHost()
    n = rows.shape[1]
    cols = np.arange(n) if n <= DUMP_SURFELS else np.sort(np.random.default_rng(0).choice(n, DUMP_SURFELS, replace=False))
    out = {"keyframe_poses": poses.astype(np.float32), "keyframe_activations": act.astype(np.float64),
           "ba_result": np.array([getattr(res, f) for f in DUMP_RESULT_FIELDS], np.float64),
           "surfel_rows": np.ascontiguousarray(rows[:8, cols], np.float32), "surfel_active": flags[cols].astype(np.float32),
           "surfel_index": cols.astype(np.float64)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def check_replicas(scene, ba, step, dev, rank, world):
    """Correctness of the N-rank step, carried by the bench line: (1) after one more (untimed) step every rank's replica --
    surfel rows, active flags, keyframe poses and activations -- must be bit-identical (hashes all-gathered); (2) rank 0 runs
    the same step on ONE GPU (a world-size-1 backend on its device) and reports the difference of the N-rank result to it."""
    import hashlib
    import torch
    import torch.distributed as dist
    from badslam_b200.direct_ba import DirectBA
    from badslam_b200.scene import pose_error
    step()
    torch.cuda.synchronize()
    rows, flags = ba.GetSurfelsHost(), ba.GetActiveHost()
    poses, act = ba.GetKeyframeStates()
    digest = hashlib.sha256(rows.tobytes() + flags.tobytes() + np.ascontiguousarray(poses).tobytes() + np.ascontiguousarray(act).tobytes()).digest()
    mine = torch.tensor(list(digest), dtype=torch.uint8, device=dev)
    gathered = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(gathered, mine)
    identical = all(bool(torch.equal(g, gathered[0])) for g in gathered)
    out = {"replicas_bit_identical": identical, "ranks": world}
    if rank == 0:
        single = DirectBA.from_scene(scene, device=dev)
        single.SetLastBAIterationCount(single.ba_iteration_count())
        single.BundleAdjustment(None, False, False, False, True, True, 1, 1, increase_ba_iteration_count=False)
        torch.cuda.synchronize()
        rows1, flags1 = single.GetSurfelsHost(), single.GetActiveHost()
        poses1, act1 = single.GetKeyframeStates()
        errs = [pose_error(poses[k], poses1[k]) for k in range(scene.cfg.num_keyframes)]
        out.update({"vs_1gpu_pose_max_m": float(max(e[0] for e in errs)), "vs_1gpu_pose_max_rad": float(max(e[1] for e in errs)),
                    "vs_1gpu_surfel_rows_max_abs": float(np.max(np.abs(rows[:8].astype(np.float64) - rows1[:8].astype(np.float64))[[0, 1, 2, 6, 7]])),
                    "vs_1gpu_packed_normals_differ": int((rows[3].view(np.uint32) != rows1[3].view(np.uint32)).sum()),
                    "vs_1gpu_active_flags_equal": bool(np.array_equal(flags, flags1)),
                    "vs_1gpu_keyframe_activations_equal": bool(np.array_equal(act, act1)),
                    "tolerance": "north_star: 1e-5 m / 1e-5 rad on poses"})
        del single
        torch.cuda.empty_cache()
    dist.barrier(device_ids=[dev.index])
    return out


def run_e2e(args, scene, dev, residuals, all_keyframes=False):
    """all_keyframes=False: the streaming case -- ONE new keyframe's RGB-D images arrive per BA call (the other keyframes are
    already resident, as in BadSlam where every keyframe is uploaded once).  all_keyframes=True: every keyframe's images are
    re-uploaded from pinned host memory in every step (nothing image-like is resident when the step starts)."""
    import torch
    from badslam_b200.direct_ba import DirectBA
    K = scene.cfg.num_keyframes
    ba = DirectBA.from_scene(scene, device=dev, host_owned=True)
    surf = ba.SurfelsDeviceView()
    backup = surf[:8].clone()
    poses0 = scene.poses_init.copy()
    act0 = np.zeros(K, np.int32)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int16 if a.dtype == np.uint16 else a.dtype)).pin_memory()
    slots = K if all_keyframes else min(K, 4)
    pinned = [(pin(scene.depth[k]), pin(scene.normals[k]), pin(scene.radius[k]), pin(scene.color[k])) for k in range(slots)]
    per_kf = sum(t.numel() * t.element_size() for t in pinned[0])
    h2d = (K if all_keyframes else 1) * per_kf + K * (96 + 28 + 4)
    d2h = K * (28 + 4 + 4 + 64)

    ba.SetLastBAIterationCount(ba.ba_iteration_count())   # (see run_ours: no end-of-scheme maintenance inside a step)

    def step(i):
        for k in (range(K) if all_keyframes else (i % slots,)):
            d, n, r, c = pinned[k]
            ba.UpdateKeyframeHost(k, d, n, r, c)
        surf[:8].copy_(backup, non_blocking=True)
        ba.SetKeyframeStates(poses0, act0)
        res = ba.BundleAdjustment(None, False, False, False, True, True, 1, 1, increase_ba_iteration_count=False)
        ba.GetKeyframeStates()
        return res

    steps = min(args.steps, 3) if all_keyframes else args.steps
    for i in range(1 if all_keyframes else max(args.warmup, 1)):
        step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        step(i)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    del ba
    return {"value": residuals / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": int(d2h), "steps": steps,
            "variant": ("every keyframe's RGB-D images re-uploaded every step" if all_keyframes else
                        "one new keyframe per BA call (streaming: the other keyframes' images are already resident)"),
            "path": "badslam_b200.DirectBA (C ABI *_host entry points): keyframe RGB-D images from pinned host memory + poses H2D, "
                    "BundleAdjustment(1 iteration), poses/activations/statistics D2H"}


def run_e2e_multi(args, scene, dev, residuals, rank, world):
    """e2e at N > 1: every rank drives its replica through the host-buffer entry points; time = max over ranks."""
    import torch
    import torch.distributed as dist
    from badslam_b200.direct_ba import DirectBA
    K = scene.cfg.num_keyframes
    ba = DirectBA.from_scene(scene, device=dev, host_owned=True, rank=rank, world_size=world)
    ba.SetCollective()
    surf = ba.SurfelsDeviceView()
    backup = surf[:8].clone()
    poses0 = scene.poses_init.copy()
    act0 = np.zeros(K, np.int32)
    ba.SetLastBAIterationCount(ba.ba_iteration_count())
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int16 if a.dtype == np.uint16 else a.dtype)).pin_memory()
    slots = min(K, 4)
    pinned = [(pin(scene.depth[k]), pin(scene.normals[k]), pin(scene.radius[k]), pin(scene.color[k])) for k in range(slots)]
    h2d = sum(t.numel() * t.element_size() for t in pinned[0]) + K * (96 + 28 + 4)
    d2h = K * 17 * 4

    def step(i):
        d, n, r, c = pinned[i % slots]
        ba.UpdateKeyframeHost(i % slots, d, n, r, c)
        surf[:8].copy_(backup, non_blocking=True)
        ba.SetKeyframeStates(poses0, act0)
        ba.BundleAdjustment(None, False, False, False, True, True, 1, 1, increase_ba_iteration_count=False)
        ba.GetKeyframeStates()

    for i in range(3):
        step(i)
    dist.barrier(device_ids=[dev.index])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    torch.cuda.synchronize()
    dist.barrier(device_ids=[dev.index])
    dt = torch.tensor([(time.perf_counter() - t0) / args.steps], device=dev, dtype=torch.float64)
    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    dt = float(dt.item())
    del ba
    return {"value": residuals / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "h2d_bytes_per_step": int(h2d * world),
            "d2h_bytes_per_step": int(d2h * world),
            "path": "badslam_b200.DirectBA per rank (C ABI *_host entry points) + torch.distributed NCCL exchange"}


def run_reference(args, scene):
    """The reference's own CUDA kernels (oracle/_ref) on one GPU, through the restated host loop."""
    import torch
    from oracle import ref_cuda
    K = scene.cfg.num_keyframes
    if not ref_cuda.available():
        # reference CUDA not usable -> time the CPU port of the reference path instead
        cb = cpu_port_baseline(scene)
        return {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": 1, "steps": 1, "warmup": 0,
                "higher_is_better": True, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "config": {"workload": scene.cfg.name}}
    ref = ref_cuda.RefDirectBA(scene)
    ref.snapshot()
    # --intrinsics (cfg4): OptimizeIntrinsicsCUDA for the depth camera + depth deformation and the colour camera inside the
    # iteration (direct_ba_alternating.cc:599-655), camera model restored before every step like on our arm
    intr = bool(getattr(args, "intrinsics", False))
    kw = dict(optimize_depth_intrinsics=intr, optimize_color_intrinsics=intr)
    if intr:
        d0, c0, a0 = ref.intrinsics()
        cf0 = ref.cfactor()
    _restore = ref.restore

    def restore():
        _restore()
        if intr:
            ref.set_intrinsics(d0, c0)
            ref.set_depth_params(a0, cf0)
    ref.restore = restore
    # residual count from the reference's own debug counters (untimed): n_count = n_assoc + n_photo with both residual types,
    # n_depth_count = n_assoc from the same launches with the descriptor residuals off.  Our metric counts both descriptor
    # residuals of a pair: n_assoc + 2 n_photo = 2 n_count - n_depth_count.  (This arm loads nothing of the product.)
    r = ref.bundle_adjust(True, True, 1, 1, count_residuals=2, end_tasks=False)
    count_ref, count_depth = int(r.n_count), int(r.n_depth_count)
    residuals = args.residuals_override or (2 * count_ref - count_depth)
    for _ in range(max(args.warmup - 1, 0)):
        ref.restore()
        ref.bundle_adjust(True, True, 1, 1, count_residuals=False, end_tasks=False, **kw)
    ref.sync()
    sampler = ClockSampler(0)
    sampler.start()
    launches0 = ref.launch_count()
    t0 = time.perf_counter()
    stage = np.zeros(3)
    for _ in range(args.steps):
        ref.restore()
        r = ref.bundle_adjust(True, True, 1, 1, count_residuals=False, end_tasks=False, **kw)
        stage += [r.ms_surfel_activation, r.ms_geometry_optimization, r.ms_pose_optimization]
    ref.sync()
    dt = (time.perf_counter() - t0) / args.steps
    clocks = sampler.stop()
    launches = ref.launch_count() - launches0
    # second headline: one full BundleAdjustment call (10 iterations + PerformBASchemeEndTasks), wall time like our arm
    ref.restore()
    ref.sync()
    t0 = time.perf_counter()
    full = ref.bundle_adjust(True, True, 10, 10, count_residuals=False, end_tasks=True, **kw)
    ref.sync()
    ms_full = (time.perf_counter() - t0) * 1e3
    value = residuals / dt
    extra_cfg = {"intrinsics": "depth intrinsics + depth deformation + colour intrinsics optimised in every step (--intrinsics)"} if intr else {}
    return {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(scene), "keyframes": K, "surfels": scene.num_surfels,
                       "residuals_per_step": int(residuals),
                       "l2": "inputs larger than L2 (keyframe images + surfels)", "parallelism": "gpus=1", **extra_cfg},
            "residual_count_source": "the reference's own debug counters (kernel_opt_pose.cu:312-320,373-381): one untimed iteration "
                                     "with both residual types (n_assoc + n_photo) and the same launches with the descriptor "
                                     "residuals off (n_assoc); residuals = n_assoc + 2 n_photo",
            "reference_debug_count": count_ref, "reference_depth_count": count_depth,
            "ms_full_ba_10_iterations": ms_full, "full_ba_iterations": int(full.iterations_done),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "reference",
                             "sample": "the reference's own unmodified CUDA kernels (oracle/_ref, built for sm_100 with its own flags) on "
                                       "ONE B200, driven by one host thread through the restated DirectBA host loop; the reference has "
                                       "no CPU implementation of this path"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": int(launches), "clocks": clocks,
            "stage_ms": {"BA_surfel_activation": stage[0] / args.steps, "BA_geometry_optimization": stage[1] / args.steps,
                         "BA_pose_optimization": stage[2] / args.steps}}


def load_scene(workload, rank, world, wait_seconds=1800):
    """The seeded scene of `workload`.  With one process per GPU, rank 0 generates it once and the other ranks load its pickle
    (BADBA_SCENE_CACHE, a per-job directory under /tmp unless set) instead of every rank spending a host-core-minute on the same
    numpy work; a rank that waited in vain generates the scene itself (it is deterministic)."""
    from badslam_b200.scene import config_by_name, make_scene, scene_cache_path
    cfg = config_by_name(workload)
    if world > 1:
        cache = os.environ.setdefault("BADBA_SCENE_CACHE", os.path.join(
            "/tmp", f"badba_scenes_{os.environ.get('MASTER_PORT', '0')}_{os.environ.get('TORCHELASTIC_RUN_ID', 'run')}"))
        path = scene_cache_path(cfg, cache)
        if rank != 0:
            t_wait = time.time()
            while not os.path.exists(path) and time.time() - t_wait < wait_seconds:
                time.sleep(0.2)
    return make_scene(cfg)


def main():
    # Exactly one JSON line may reach stdout: route everything libraries print there (e.g. NCCL's version banner)
    # to stderr while the benchmark runs.
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        return _main(saved_stdout)
    finally:
        try:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


def _main(saved_stdout):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("BADBA_WORKLOAD", "cfg3"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e-all", action="store_true", help="skip the e2e variant that re-uploads every keyframe every step")
    ap.add_argument("--intrinsics", action="store_true",
                    help="optimise depth intrinsics + depth deformation and colour intrinsics inside the step (the cfg4 configuration)")
    ap.add_argument("--residuals-override", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))

    from badslam_b200.scene import config_by_name, make_scene
    if args.impl == "reference" and rank != 0:
        return 0
    scene = load_scene(args.workload, rank, world)
    if args.impl == "reference":
        out = run_reference(args, scene)
    else:
        out = run_ours(args, scene, rank, world)
    if rank == 0:
        sys.stdout.flush()
        os.write(saved_stdout, (json.dumps(out) + "\n").encode())
    return 0


if __name__ == "__main__":
    sys.exit(main())
