#!/usr/bin/env python
"""Benchmark of the per-frame perception hot path (BASELINE.json: points/s & frames/s per B200).

A "step" = one pass of the whole hot path (crop -> VoxelGrid -> RANSAC plane loop -> Euclidean clustering ->
centroid/radius) over one batch of synthetic HDL-64-style 120 000-point frames (BASELINE.json configs[1],
parameters of SURVEY.md 8d config 2), `--batch` frames per GPU per step, through the C ABI (one pcop_process_batch
call per step).

  value     points/s, whole job: frames already resident in HBM (the batch, 1.97 GB at 1024 frames, is larger than
            the 126 MB L2, so every step re-reads its input from HBM; no explicit L2 flush), EVERY requested result
            array delivered to pinned host memory inside the step (the boundary's semantics, SURVEY 8b)
  e2e       the same with HOST (pinned) frames: H2D of the frames and D2H of the results inside the timed region
  roofline  SURVEY 8(d) figure of the dominant STAGE: algorithmic bytes of the stage / its device time, measured live
            with CUDA events on the library's stream (a second pass of the same K steps); `pipeline_roofline` is the
            whole pipeline, `stages` every stage, `kernels` every kernel (scratch-inclusive traffic efficiency)
  configs   BASELINE.json configs[0], [2], [3] (single-frame latency + a small batch) and configs[4] (4096 frames
            per GPU per step in one call)
  cpu_baseline  the CPU oracle (PCL-semantics restatement, oracle/) on a bounded sample of the same frames
  N > 1     frames sharded over the ranks (weak scaling), times = the slowest rank's; `per_rank_ms_per_step` lists every
            rank; `value` adds the gather of cluster_offsets / cluster_indices / obstacles to rank 0 over NCCL (SURVEY
            8e), `value_results_left_in_hbm_gathered` is the same gather with the arrays left in HBM on every rank,
            `host_path` / `d2h_GBps_aggregate` say what the box's host path allows
  clocks    SM clock + throttle reasons from NVML, sampled every 4 ms inside the timed region (rank 0)

`--impl reference` times that CPU restatement with all host threads on the same config (the reference itself needs
ROS + PCL and cannot be built in this image; see DESIGN.md).

`--dump-outputs DIR` writes what the last timed step returned (rank 0's frames) as DIR/<name>.npy, see dump_outputs();
the frames are generated from fixed seeds, so two builds run with the same arguments can be compared file for file.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIG = 2  # BASELINE.json configs[1]: HDL-64-style 120k-point frame
METRIC = "points/sec per B200 job (HDL-64 120k-point frames: crop + 0.1 m voxel + RANSAC ground removal + Euclidean clustering + centroid/radius)"


def workload_config(n, batch, world):
    """`config` of the JSON line; identical for both arms (--impl ours / reference)."""
    return {"workload": "BASELINE configs[1]: HDL-64-style 120k-point frame, crop + 0.1 m voxel + ground-plane RANSAC + "
                        "Euclidean clustering + centroid/radius (SURVEY 8d config 2 parameters)",
            "points_per_frame": n, "frames_per_gpu_per_step": batch,
            "parallelism": f"frames sharded over {world} GPU(s), no intra-frame collective"}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """SM clock + throttle reasons during the timed region (B200_PROFILING.md recipe).  The values are NVML's -- what
    nvidia-smi prints -- read in-process every few milliseconds (the timed region lasts tens of milliseconds; spawning
    nvidia-smi takes longer than that and competes with the engine's host thread for the rank's cores).  Falls back to
    the nvidia-smi command line when the NVML binding is missing.  `active` = False: no sampling (ranks other than 0)."""

    def __init__(self, gpu_index, active=True):
        self.gpu = gpu_index
        self.active = active
        self.rows = []
        self.source = None
        self._stop = threading.Event()
        self._t = None

    def _run_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        masks = ((8, "hw_slowdown"), (64, "hw_thermal_slowdown"), (32, "sw_thermal_slowdown"), (4, "sw_power_cap"))
        self.source = "nvml"
        self._ready.set()
        while not self._stop.is_set():
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.rows.append([str(sm), str(mx)] + [("Active" if r & m else "Not Active") for m, _ in masks])
            self._stop.wait(0.004)

    def _run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            self.source = "nvidia-smi"
            self._ready.set()
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                parts = [x.strip() for x in out.stdout.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        if self.active:
            self._ready = threading.Event()
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
            self._ready.wait(timeout=10)  # (NVML initialised before the timed region starts)
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=6)

    def summary(self):
        sm = []
        reasons = set()
        mx = None
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": self.source}


def oracle_frames_per_sec(params, frames, threads):
    """CPU oracle over `frames` ([F, n, 4]) with `threads` host threads; returns (frames/s, seconds)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    O.lib()
    t0 = time.perf_counter()
    if threads <= 1:
        for f in range(len(frames)):
            O.process(params, frames[f])
    else:
        with ThreadPoolExecutor(max_workers=threads) as ex:
            list(ex.map(lambda f: O.process(params, frames[f]), range(len(frames))))
    dt = time.perf_counter() - t0
    return len(frames) / dt, dt


def run_reference(args, rank, world, emit):
    """--impl reference: the CPU restatement (oracle port) with all host threads; same metric, config and frames per
    step as the other arm (1024 frames take about a second per step on 16 threads)."""
    if rank != 0:
        return
    from pointcloud_obstacle_processing_b200 import synth
    n = synth.points_per_frame(CONFIG)
    threads = os.cpu_count() or 1
    frames = synth.frames(CONFIG, 0, args.batch)
    params = synth.params(CONFIG)
    for _ in range(min(args.warmup, 1)):
        oracle_frames_per_sec(params, frames[:2 * threads], threads)
    times = []
    for _ in range(args.steps):
        _, dt = oracle_frames_per_sec(params, frames, threads)
        times.append(dt)
    total = sum(times)
    fps = args.steps * args.batch / total
    pps = fps * n
    line = {
        "impl": "reference", "metric": METRIC, "value": pps, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(n, args.batch, world),
        "frames_per_sec": fps,
        "cpu_baseline": {"value": pps, "unit": "points/s", "cores": threads, "kind": "port",
                         "sample": f"{args.batch} synthetic config-2 frames per step (the other arm's batch), "
                                   f"frame-parallel over {threads} host threads; PCL-semantics CPU restatement "
                                   f"(oracle/), not PCL itself; one warm-up pass over {2 * threads} frames"},
        "e2e": {"value": pps, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def frame_alg_bytes(p, r):
    """SURVEY 8(d) algorithmic bytes of one frame result, per stage group."""
    b = {"crop+voxel": 0.0, "sor": 0.0, "plane": 0.0, "cluster+centroid": 0.0}
    if p.enable_crop:
        b["crop+voxel"] += 16.0 * r.n_input + 20.0 * r.n_crop
    if p.enable_voxel:
        b["crop+voxel"] += 16.0 * r.n_crop + 20.0 * r.n_voxel
    if p.enable_sor:
        b["sor"] += 16.0 * r.n_voxel + 20.0 * r.n_sor
    if p.enable_plane:
        pk = r.n_sor
        for k in range(min(r.n_plane_passes, len(r.plane_pass_inliers))):
            ik = r.plane_pass_inliers[k]
            b["plane"] += 16.0 * pk + 16.0 * (pk - ik) + 4.0 * ik + 16.0
            pk -= ik
    if p.enable_cluster:
        b["cluster+centroid"] += 32.0 * r.n_remaining + 8.0 * r.n_cluster_points + 4.0 * (r.n_clusters + 1) + 16.0 * r.n_clusters
    return b


DUMP_FRAMES = 256        # frames of the batch whose result arrays --dump-outputs writes
DUMP_LIMIT = 64 << 20    # bytes of all --dump-outputs files together
SCALAR_FIELDS = ("status", "warnings", "n_input", "n_crop", "n_voxel", "n_sor", "n_remaining", "n_clusters",
                 "n_cluster_points", "n_plane_passes", "n_plane_inliers")
ARRAY_FIELDS = ("crop_kept_idx", "voxel_keys", "voxel_centroids", "sor_kept_idx", "plane_inlier_idx", "remaining_cloud",
                "remaining_src_idx", "cluster_offsets", "cluster_indices", "obstacles")


def dump_outputs(res, out_dir):
    """Writes the host results of one pcop_process_batch call (`res`, its ctypes result array) to out_dir/<field>.npy.

    Every frame: the counts and warnings (float64 [B]) and the plane records (plane_pass_points / plane_pass_inliers
    float64 [B, 16], plane_pass_coeff float32 [B, 16, 4], zero past n_plane_passes; plane_coeff float32 [B, 4]).
    The result arrays of a fixed sample of frames (seed 0, ascending, listed in frame_index.npy) are concatenated in
    that order -- the frame's count fields split them: float arrays stay float32, index arrays become float64 (exact).
    Frames are dropped from the end of the sample if all files together would exceed DUMP_LIMIT bytes."""
    from pointcloud_obstacle_processing_b200 import Frame
    from pointcloud_obstacle_processing_b200._ctypes_abi import MAX_PASSES
    B = len(res)
    out = {k: np.array([getattr(r, k) for r in res], np.float64) for k in SCALAR_FIELDS}
    out["plane_pass_points"] = np.zeros((B, MAX_PASSES), np.float64)
    out["plane_pass_inliers"] = np.zeros((B, MAX_PASSES), np.float64)
    out["plane_pass_coeff"] = np.zeros((B, MAX_PASSES, 4), np.float32)
    out["plane_coeff"] = np.zeros((B, 4), np.float32)
    frames = {}
    for k, r in enumerate(res):
        f = Frame.from_c(r)
        npass = len(f.plane_pass_points)
        out["plane_pass_points"][k, :npass] = f.plane_pass_points
        out["plane_pass_inliers"][k, :npass] = f.plane_pass_inliers
        out["plane_pass_coeff"][k, :npass] = f.plane_pass_coeff
        out["plane_coeff"][k] = f.plane_coeff
        frames[k] = f
    sample = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_FRAMES), replace=False))
    budget = DUMP_LIMIT - sum(a.nbytes for a in out.values()) - sample.size * 8 - 128 * (len(out) + len(ARRAY_FIELDS) + 1)
    parts = {k: [] for k in ARRAY_FIELDS}
    kept = []
    for k in sample:
        arrays = {name: getattr(frames[k], name) for name in ARRAY_FIELDS if getattr(frames[k], name) is not None}
        arrays = {name: a if a.dtype == np.float32 else a.astype(np.float64) for name, a in arrays.items()}
        size = sum(a.nbytes for a in arrays.values())
        if size > budget:
            break
        budget -= size
        kept.append(k)
        for name, a in arrays.items():
            parts[name].append(a)
    out["frame_index"] = np.array(kept, np.float64)
    for name, p in parts.items():
        if p:
            out[name] = np.concatenate(p)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def small_config(cfg, batch, reps, local_rank, peak, torch):
    """BASELINE configs[0] / [2] / [3]: single-frame latency (host in -> results on host) and a small device-resident
    batch, with its SURVEY 8(d) fraction."""
    from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
    n = synth.points_per_frame(cfg)
    p = synth.params(cfg)
    host = torch.empty((batch, n, 4), dtype=torch.float32).pin_memory()
    synth.frames(cfg, 0, batch, out=host.numpy())
    dev = host.to(f"cuda:{local_rank}")
    counts = np.full(batch, n, np.int32)
    out = {"points_per_frame": n, "batch": batch}
    with ObstacleProcessor(p, n, max_batch=1, device=local_rank) as op1:
        for _ in range(5):
            op1.process_batch_raw(host.data_ptr(), n, counts[:1])
        ts = []
        for i in range(reps):
            a = time.perf_counter()
            op1.process_batch_raw(host.data_ptr() + (i % batch) * n * 16, n, counts[:1])
            ts.append((time.perf_counter() - a) * 1e3)
        ts.sort()
        out["p50_ms"] = ts[len(ts) // 2]
        out["launches_per_frame"] = int(op1.last_launch_count)
    with ObstacleProcessor(p, n, max_batch=batch, device=local_rank) as op:
        for _ in range(3):
            res = op.process_batch_raw(dev.data_ptr(), n, counts)
        torch.cuda.synchronize()
        steps = 5
        t0 = time.perf_counter()
        for _ in range(steps):
            res = op.process_batch_raw(dev.data_ptr(), n, counts)
        dt = (time.perf_counter() - t0) / steps
        alg = op.last_algorithmic_bytes
        out.update({"points_per_sec": batch * n / dt, "frames_per_sec": batch / dt, "ms_per_step": dt * 1e3,
                    "roofline_frac": alg / dt / 1e9 / peak,
                    "counts_frame0": {k: int(getattr(res[0], k)) for k in ("n_crop", "n_voxel", "n_remaining", "n_clusters")}})
    del dev, host
    torch.cuda.empty_cache()
    return out


# What the numbers at N > 1 run into on the pool's 8-GPU boxes, measured with tools/pcie_probe.sh and
# tools/n8_sync_probe.py (profiles/pcie_probe_r02_n8.txt, profiles/n8_sync_probe_r02.txt):
HOST_PATH_NOTE = ("result delivery to the host is bound by the box, not by the GPUs: with 8 GPUs copying device-to-host at once "
                  "the box sustains 113 GB/s in total (4 GPUs at 8.8 GB/s, 4 at 19.4 GB/s; one GPU alone 56 GB/s), while 8 "
                  "ranks at single-GPU speed need 8 x 22 GB/s.  With the results left in HBM and the ranks barrier-aligned "
                  "(no gather) six of the eight ranks run the 1024-frame call in 5.15-5.25 ms, the single-GPU time, and two "
                  "(ranks 3 and 6: same on two boxes, pinned or unpinned host threads, 3 or 4 lanes, 1965 MHz, no throttle "
                  "reason; rank 3 of a 4-GPU job as well) take 6.5 ms, although GPU 3 runs the same call in 5.2 ms in a "
                  "process of its own -- cause not identified; the line's time is the slowest rank's, "
                  "`per_rank_ms_per_step` lists them all")


def main():
    # the contract is ONE JSON line on stdout: everything else that libraries print there (NCCL's version banner,
    # ...) is sent to stderr; emit() writes to the real stdout
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="frames per GPU per step")
    ap.add_argument("--latency-reps", type=int, default=200)
    ap.add_argument("--cpu-sample", type=int, default=128, help="frames of the CPU-baseline sample")
    ap.add_argument("--no-kernel-timing", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs[0], [2], [3], [4] section")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world, emit)
        return

    import torch
    import torch.distributed as dist
    from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        try:  # one rank per GPU; the box's hardware threads are shared out so that the ranks' host threads do not migrate
            ncpu = os.cpu_count() or 1
            per = max(1, ncpu // world)
            os.sched_setaffinity(0, set(range(local_rank * per, min(ncpu, (local_rank + 1) * per))))
        except Exception:
            pass
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n = synth.points_per_frame(CONFIG)
    B = args.batch
    params = synth.params(CONFIG)
    # distinct frames per rank (weak scaling: per-GPU work fixed)
    host = torch.empty((B, n, 4), dtype=torch.float32).pin_memory()
    synth.frames(CONFIG, rank * B, B, out=host.numpy())
    dev = host.to(f"cuda:{local_rank}", non_blocking=False)
    counts = np.full(B, n, np.int32)
    from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi
    op = ObstacleProcessor(params, n, max_batch=B, device=local_rank)

    def step_device():
        return op.process_batch_raw(dev.data_ptr(), n, counts)

    def step_host():
        return op.process_batch_raw(host.data_ptr(), n, counts)

    # ---- final result gather (SURVEY 8e), once per step: cluster_offsets, cluster_indices and obstacles of every frame
    # to rank 0 over NCCL (sizes first, then the three arrays padded to a fixed per-rank capacity).  Asynchronous and
    # double-buffered: the collectives of step k run on NCCL's stream while step k+1 computes; flush() waits for the
    # outstanding ones before a timed region ends.
    gather = sharding.ResultGather(B, torch.device("cuda", local_rank)) if world > 1 else None
    # The staging of step k's arrays (a few dozen asynchronous copies out of the library's pinned result buffer) and the
    # launch of its collectives run on a helper thread while the main thread is already inside the library call of step
    # k + 1 (the library keeps a call's results valid while the next call runs, so at most one step may be pending).
    import queue
    gq = queue.Queue(maxsize=1)
    gerr = []

    def gather_worker():
        torch.cuda.set_device(local_rank)
        while True:
            item = gq.get()
            if item is None:
                gq.task_done()
                return
            try:
                gather.submit(item)
            except Exception as e:  # surfaced by gather_flush()
                gerr.append(e)
            gq.task_done()

    gthread = None
    if gather is not None and not os.environ.get("PCOP_BENCH_NO_GATHER"):
        gthread = threading.Thread(target=gather_worker, daemon=True)
        gthread.start()

    def gather_results(res):
        if gthread is not None:
            gq.join()      # the previous step's staging has been enqueued ...
            gather.wait_staged()  # ... and has run: its result buffer is free for the call after this one
            gq.put(res)

    def gather_flush():
        if gthread is not None:
            gq.join()
            if gerr:
                raise gerr[0]
            gather.flush()

    peak, peak_kind = measured_peak_gbs()
    # ---- headline: frames resident in HBM, every result array delivered to pinned host memory ------------------------
    for _ in range(max(args.warmup, 3)):
        gather_results(step_device())
    gather_flush()
    launches = 0
    alg_bytes = 0.0
    dev_us = 0.0
    with ClockSampler(local_rank, active=(rank == 0)) as clocks:
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = step_device()
            gather_results(res)
            dev_us += op.last_elapsed_us
            launches += op.last_launch_count
            alg_bytes += op.last_algorithmic_bytes
        gather_flush()
        torch.cuda.synchronize()
        own_wall = time.perf_counter() - t0  # this rank's own K steps (the line's time is the slowest rank's)
        barrier()
        wall = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:  # (before the next call on the handle reuses the result buffers)
        dump_outputs(res, args.dump_outputs)
    stage_alg = {}
    for r in res:
        for k, v in frame_alg_bytes(params, r).items():
            stage_alg[k] = stage_alg.get(k, 0.0) + v
    counts_sum = {k: sum(getattr(r, k) for r in res) for k in
                  ("n_input", "n_crop", "n_voxel", "n_remaining", "n_clusters", "n_cluster_points")}
    plane_passes = sum(r.n_plane_passes for r in res)

    # ---- extra: the same K steps with the result arrays LEFT in HBM (outputs | OUT_DEVICE: device pointers for a
    # GPU-side consumer; counts, warnings and plane records still reach the host) -------------------------------------
    params_dev = params.copy()
    params_dev.outputs = abi.OUT_DEFAULT | abi.OUT_DEVICE
    op.set_params(params_dev)
    for _ in range(2):
        step_device()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_device()
    torch.cuda.synchronize()
    own_wall_dev = time.perf_counter() - t0
    barrier()
    wall_dev_results = time.perf_counter() - t0

    def per_rank_ms(own):
        """ms per step of every rank's own K steps (rank order); None on one GPU"""
        if world == 1:
            return None
        t = torch.tensor([1000.0 * own / args.steps], dtype=torch.float64, device=dev.device)
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [round(float(x.item()), 3) for x in out]

    per_rank = {"results_to_host": per_rank_ms(own_wall), "results_left_in_hbm": per_rank_ms(own_wall_dev)}

    # ---- extra (N > 1): SURVEY 8(e) as written -- the result arrays stay in HBM and cluster_offsets / cluster_indices /
    # obstacles of every rank go to rank 0 over NCCL straight from the library's device result buffer (no host copy of
    # the arrays on any rank).  The staging of a step's arrays has to finish before the next call reuses the buffer, so
    # it runs on the main thread here (a few dozen device-to-device copies).
    gathered_dev = None
    if gather is not None and gthread is not None:
        for _ in range(2):
            gather.submit(step_device())
            gather.wait_staged()
        gather.flush()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            gather.submit(step_device())
            gather.wait_staged()
        gather.flush()
        torch.cuda.synchronize()
        own_wall_gd = time.perf_counter() - t0
        barrier()
        wall_gd = time.perf_counter() - t0
        per_rank["results_left_in_hbm_gathered"] = per_rank_ms(own_wall_gd)
        gathered_dev = {"value": world * args.steps * B * n / wall_gd, "unit": "points/s", "ms_per_step": 1000.0 * wall_gd / args.steps,
                        "gather_bytes_per_rank_per_step": int(gather.bytes_per_step),
                        "what": "SURVEY 8(e) as written: result arrays left in HBM on every rank, cluster_offsets / cluster_indices / "
                                "obstacles of all ranks gathered to rank 0 over NCCL straight from the device result buffers"}
    op.set_params(params)

    # ---- instrumented pass: the same K steps with a CUDA-event pair around every launch and every stage on the
    # library's stream.  Per-kernel timing needs each kernel alone on the GPU, so the library serialises its lanes
    # here; this pass feeds `roofline`, `stages`, `kernels` only, never `value`.
    kernel_times = {}
    stage_acc = {}
    wall_instr = None
    if not args.no_kernel_timing:
        # (its own handle: ONE lane with 256-frame waves -- the three lanes of the timed runs keep 3 x 128 frames in
        # flight, a single lane of 128-frame waves would leave the latency-bound kernels a third of that)
        saved = {k: os.environ.get(k) for k in ("PCOP_LANES", "PCOP_WAVE_FRAMES")}
        os.environ["PCOP_LANES"] = "1"
        os.environ["PCOP_WAVE_FRAMES"] = str(min(256, B))
        op_i = ObstacleProcessor(params, n, max_batch=B, device=local_rank)
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        op_i.process_batch_raw(dev.data_ptr(), n, counts)  # untimed: grows the pinned result buffer, adapts the grids
        op_i.enable_kernel_timing(True)
        op_i.process_batch_raw(dev.data_ptr(), n, counts)
        op_i.enable_kernel_timing(True)  # (re-enabling clears the accumulated totals)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            op_i.process_batch_raw(dev.data_ptr(), n, counts)
            for k, v in op_i.stage_times_us().items():
                stage_acc[k] = stage_acc.get(k, 0.0) + v
        barrier()
        wall_instr = time.perf_counter() - t0
        kernel_times = op_i.kernel_times()
        op_i.close()

    # ---- end-to-end run (host frames in, results out) ------------------------------------------------
    for _ in range(2):
        step_host()
    barrier()
    t1 = time.perf_counter()
    d2h_exact = 0.0
    for _ in range(args.steps):
        gather_results(step_host())
        d2h_exact += op.last_d2h_bytes
    gather_flush()
    barrier()
    wall_e2e = time.perf_counter() - t1
    d2h_bytes = d2h_exact / args.steps  # counted by the library from the copies it issued

    # ---- max over ranks -----------------------------------------------------------------------------
    t = torch.tensor([wall, wall_e2e, dev_us * 1e-6, wall_dev_results], dtype=torch.float64, device=dev.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall, wall_e2e, dev_s, wall_dev_results = [float(x) for x in t.tolist()]

    # ---- BASELINE configs[4]: 4096 frames per GPU per step, ONE pcop_process_batch call per step (the handle keeps
    # max_batch = B frames of wave buffers; the call runs 4096 / wave frames waves).  The 4096 frames are the step's B
    # distinct frames repeated (7.86 GB resident in HBM).
    cfg5 = None
    if not args.no_configs:
        reps5 = max(1, 4096 // B)
        big = dev.repeat(reps5, 1, 1) if reps5 > 1 else dev
        nb = big.shape[0]
        counts5 = np.full(nb, n, np.int32)
        for _ in range(2):  # (both of the handle's alternating pinned result buffers grow to the call's size here)
            op.process_batch_raw(big.data_ptr(), n, counts5)
        barrier()
        t0 = time.perf_counter()
        steps5 = 2
        for _ in range(steps5):
            op.process_batch_raw(big.data_ptr(), n, counts5)
        barrier()
        w5 = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev.device)
        if world > 1:
            dist.all_reduce(w5, op=dist.ReduceOp.MAX)
        w5 = float(w5.item())
        cfg5 = {"frames_per_gpu_per_step": nb, "calls_per_step": 1, "steps": steps5,
                "points_per_sec": world * steps5 * nb * n / w5, "frames_per_sec": world * steps5 * nb / w5,
                "ms_per_step": 1000.0 * w5 / steps5,
                "roofline_frac": (alg_bytes / (args.steps * B)) * (world * steps5 * nb) / w5 / 1e9 / (peak * world),
                "what": f"{nb} frames ({B} distinct frames x {reps5}) resident in HBM, results to pinned host memory, "
                        f"whole job over {world} GPU(s), no cross-rank gather"}
        del big
        torch.cuda.empty_cache()

    # ---- single-frame latency (rank 0) -----------------------------------------------------------------
    lat = None
    if rank == 0 and args.latency_reps > 0:
        op1 = ObstacleProcessor(params, n, max_batch=1, device=local_rank)
        for _ in range(10):
            op1.process_batch_raw(host.data_ptr(), n, counts[:1])
        ts = []
        for i in range(args.latency_reps):
            a = time.perf_counter()
            op1.process_batch_raw(host.data_ptr() + (i % B) * n * 16, n, counts[:1])
            ts.append((time.perf_counter() - a) * 1e3)
        ts.sort()
        lat = {"p50_ms": ts[len(ts) // 2], "p90_ms": ts[int(len(ts) * 0.9)], "min_ms": ts[0], "reps": len(ts),
               "launches_per_frame": int(op1.last_launch_count),
               "what": "one 120k-point frame, host pinned in -> results on host, wall clock"}
        op1.close()
    op.close()
    del dev
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs (rank 0, N = 1 only) -------------------------------------------------
    configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        configs = {}
        for key, cfg, batch in (("1", 1, 64), ("3", 3, 16), ("4", 4, 8)):
            try:
                configs[key] = small_config(cfg, batch, 50, local_rank, peak, torch)
            except Exception as e:  # (a config must not take the headline down with it)
                configs[key] = {"error": repr(e)}
        configs["1"]["what"] = "BASELINE configs[0]: VLP-16-style 30k-point frame, params.yaml verbatim (incl. SOR)"
        configs["3"]["what"] = "BASELINE configs[2]: 640x480 organized depth cloud, 0.02 m voxel, tolerance 0.05"
        configs["4"]["what"] = "BASELINE configs[3]: adversarial 1M-point frame, a few very large clusters"
    if cfg5 is not None:
        configs = configs or {}
        configs["5"] = cfg5

    # ---- CPU baseline (rank 0, N=1 only) ------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        sample = min(args.cpu_sample, B)
        fps1, dt1 = oracle_frames_per_sec(params, host.numpy()[:sample], 1)
        threads = os.cpu_count() or 1
        fpsn, dtn = oracle_frames_per_sec(params, host.numpy()[:min(B, max(sample, 2 * threads))], threads)
        cpu = {"value": fps1 * n, "unit": "points/s", "cores": 1, "kind": "port",
               "sample": f"first {sample} frames of the step's batch, single thread ({dt1:.1f} s); PCL-semantics CPU "
                         f"restatement (oracle/), the reference node is single-threaded (od.cpp:1014)",
               "frames_per_sec": fps1,
               "all_cores": {"value": fpsn * n, "unit": "points/s", "cores": threads, "frames_per_sec": fpsn}}

    if rank == 0:
        total_frames = world * args.steps * B
        total_points = total_frames * n
        value = total_points / wall
        # ---- stages and kernels, timed live -----------------------------------------------------------------
        stage_us = {"crop+voxel": stage_acc.get("crop", 0.0) + stage_acc.get("voxel", 0.0), "sor": stage_acc.get("sor", 0.0),
                    "plane": stage_acc.get("plane", 0.0),
                    "cluster+centroid": stage_acc.get("cluster", 0.0) + stage_acc.get("centroid", 0.0)}
        stages = {}
        for k, us in stage_us.items():
            if us <= 0.0 or stage_alg.get(k, 0.0) <= 0.0:
                continue
            byt = stage_alg[k] * args.steps  # (the last step's frames; every step processes the same frames)
            gbs = byt / (us * 1e-6) / 1e9
            stages[k] = {"algorithmic_bytes_per_frame": stage_alg[k] / B, "us_per_frame": us / (args.steps * B),
                         "achieved_GBps": gbs, "frac": gbs / peak}
        ktable = {}
        stage_of = {"k_vp_": "crop+voxel", "k_vf_": "crop+voxel", "k_crop": "crop+voxel", "k_voxel": "crop+voxel", "k_sort": "crop+voxel",
                    "k_plane": "plane", "k_ece": "cluster+centroid", "k_centroid": "cluster+centroid", "k_sor": "sor"}
        if kernel_times:
            tot_us = sum(v[0] for v in kernel_times.values())
            N_, M_, V_, P_ = (counts_sum[k] * args.steps for k in ("n_input", "n_crop", "n_voxel", "n_remaining"))
            L_, C_ = (counts_sum[k] * args.steps for k in ("n_cluster_points", "n_clusters"))
            # bytes each kernel moves by design (its own reads + writes INCLUDING scratch such as the partitioned
            # elements; not the SURVEY 8d figure, which is per stage): a traffic-efficiency measure per kernel
            moved = {
                "k_vp_hist": 16.0 * N_,
                "k_vp_scatter": 16.0 * N_ + 16.0 * M_,
                "k_vp_reduce": 16.0 * M_ + 16.0 * V_,
                "k_plane_loop": 16.0 * V_ + 20.0 * P_,
                "k_ece_small": 32.0 * P_ + 8.0 * L_ + 20.0 * C_,
                "k_pack": 2.0 * (20.0 * P_ + 4.0 * L_ + 20.0 * C_),
            }
            for k, (us, cnt) in sorted(kernel_times.items(), key=lambda kv: -kv[1][0]):
                e = {"total_us": round(us, 1), "launches": cnt, "avg_launch_us": round(us / max(cnt, 1), 2),
                     "share": round(us / tot_us, 4),
                     "stage": next((s for pre, s in stage_of.items() if k.startswith(pre)), "pack/other")}
                if k in moved and us > 0:
                    e["moved_GBps_scratch_inclusive"] = round(moved[k] / (us * 1e-6) / 1e9, 1)
                    e["moved_frac_of_hbm_peak"] = round(e["moved_GBps_scratch_inclusive"] / peak, 4)
                ktable[k] = e
        roof = None
        if stages:
            dom = max(stages.items(), key=lambda kv: kv[1]["us_per_frame"])
            name, st = dom
            dom_kernel = max(((k, v) for k, v in ktable.items() if v["stage"] == name), key=lambda kv: kv[1]["total_us"],
                             default=(None, None))[0]
            # DRAM bytes of the stage's kernels from the committed `ncu --set full` capture (profiles/, 256 frames per
            # launch: dram__bytes_read.sum + dram__bytes_write.sum), per frame
            # (k_vp_hist 498.6 + k_vp_scan 32.5 + k_vp_scatter 958.7 + k_vp_reduce 616.9 MB; k_plane_gen0 5.0 + k_plane_loop 246.7 MB)
            ncu_dram_per_frame = {"crop+voxel": (498.6e6 + 32.5e6 + 958.7e6 + 616.9e6) / 256.0,
                                  "plane": 251.7e6 / 256.0, "cluster+centroid": 20.9e6 / 256.0}
            roof = {"bound": "hbm", "stage": name, "kernel": dom_kernel, "achieved": st["achieved_GBps"], "peak": peak,
                    "unit": "GB/s", "frac": st["frac"],
                    "traffic": ncu_dram_per_frame.get(name, 0.0) * B if name in ncu_dram_per_frame else None,
                    "traffic_source": "profiles/ncu_full_r02c_summary.csv (ncu --set full, 256 frames per launch), scaled "
                                      "to this step's frames; per step like `algorithmic_bytes_per_step`",
                    "algorithmic_bytes_per_step": st["algorithmic_bytes_per_frame"] * B,
                    "us_per_step": st["us_per_frame"] * B, "peak_source": peak_kind,
                    "what": "SURVEY 8(d): the stage's distinct inputs read once + distinct outputs written once (sort / "
                            "partition scratch not counted) / the stage's device time; dominant stage of the step",
                    "timed": "second pass of the same K steps with CUDA-event pairs around every stage and launch on the "
                             "library's stream: one lane, 256-frame waves, so that each kernel runs alone"}
        pipe_gbs = world * alg_bytes / wall / 1e9 if wall > 0 else None
        h2d = B * n * 16 + B * 4
        line = {
            "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": 1000.0 * wall / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(n, B, world),
            "results": "every requested result array (remaining cloud + source indices, cluster CSR, obstacle records) "
                       "delivered to pinned host memory inside the step" +
                       ("; cluster_offsets / cluster_indices / obstacles of all ranks gathered to rank 0 over NCCL" if world > 1 else ""),
            "l2": "no flush: the per-step input batch (%.0f MB) exceeds the 126 MB L2" % (B * n * 16 / 1e6),
            "frames_per_sec": total_frames / wall,
            "d2h_GBps_aggregate": world * d2h_bytes / (wall / args.steps) / 1e9,
            "host_path": HOST_PATH_NOTE if world > 1 else None,
            "per_rank_ms_per_step": per_rank if world > 1 else None,
            "value_results_left_in_hbm": {"value": total_points / wall_dev_results, "unit": "points/s",
                                          "ms_per_step": 1000.0 * wall_dev_results / args.steps,
                                          "what": "same K steps with outputs | PCOP_OUT_DEVICE: result arrays stay in HBM for "
                                                  "a GPU-side consumer, only counts and plane records reach the host"},
            "value_results_left_in_hbm_gathered": gathered_dev,
            "device_ms_per_step": 1000.0 * dev_s / args.steps,
            "instrumented_ms_per_step": 1000.0 * wall_instr / args.steps if wall_instr else None,
            "e2e": {"value": total_points / wall_e2e, "unit": "points/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": int(d2h_bytes), "frames_per_sec": total_frames / wall_e2e,
                    "ms_per_step": 1000.0 * wall_e2e / args.steps,
                    "h2d_GBps_aggregate": world * h2d / (wall_e2e / args.steps) / 1e9,
                    "bound": "host-to-device copy of the frames (16 B per point over PCIe / the host memory path, shared "
                             "by the GPUs of the box)"},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            "roofline": roof,
            "pipeline_roofline": {"algorithmic_bytes_per_frame": alg_bytes / (args.steps * B),
                                  "achieved_GBps": pipe_gbs, "peak": peak * world, "frac": pipe_gbs / (peak * world) if pipe_gbs else None,
                                  "what": "sum of SURVEY 8d stage bytes over all frames of all GPUs / elapsed of the timed region "
                                          "(whole pipeline incl. result delivery); peak = measured HBM peak x GPUs"},
            "stages": stages,
            "stage_ms_per_step": {k: round(v / args.steps / 1000.0, 3) for k, v in stage_acc.items()},
            "kernels": ktable,
            "counts_per_frame": dict({k: v / B for k, v in counts_sum.items()}, plane_passes=plane_passes / B),
            "latency": lat,
            "configs": configs,
            "cpu_baseline": cpu,
        }
        emit(line)
    if gthread is not None:
        gq.put(None)
        gthread.join(timeout=10)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
