"""The occupancy-grid product of a batch: pcop_process_batch_occupancy against pcop_process_batch alone and against the
per-frame chain it replaces.

python tools/occupancy_batch_bench.py [--round r03] [--out PATH] [--frames 1024] [--rounds 7]

Per case (config 1 = params.yaml grid, config 2 at block_size 0.25 and 0.1), 1024 frames per call resident in HBM
(64 distinct frames tiled; 0.5 GB / 2 GB of input, larger than the 126 MB L2), one step = one call:
  a  pcop_process_batch alone
  b  pcop_process_batch_occupancy, grids into device memory
  c  pcop_process_batch_occupancy, grids into pinned host memory (and into a pageable numpy array, c_pageable)
  d  today's chain: pcop_process_batch, then pcop_occupancy_grid + pcop_occupancy_shadows per frame
a, b, c and c_pageable alternate within every round (the spread is the min .. max over rounds); d is slower by
orders of magnitude and runs fewer rounds.  Single-frame latency: p50 of the three-call chain against the new call with batch = 1 (host
frame in, host grid out).  A call of every case warms its shape first.  Per-kernel device times of the grid kernels
come from a separate call with kernel timing on (which serialises the lanes), so they do not enter a .. d.
Writes profiles/occupancy_batch_<round>.json (or --out)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # device memory for the resident frames and grids only

from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from shadow_util import rigid

CASES = [("config1_params_yaml", 1, None), ("config2_block_0.25", 2, 0.25), ("config2_block_0.1", 2, 0.1)]
GRID_KERNELS = ("k_occ_count_wave_s32", "k_occ_count_wave_s16", "k_occ_count_wave_g", "k_occ_threshold_wave",
                "k_occ_shadow", "k_occ_mark")


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return info


def poses(p, B, seed=1):
    rng = np.random.default_rng(seed)
    ws, sw = [], []
    for _ in range(B):
        m, inv = rigid(rng.uniform(-0.3, 0.3), rng.uniform(0.3, 0.6), 0.0,
                       [p.x_max + rng.uniform(0.2, 1.5), 0.5 * (p.y_min + p.y_max) + rng.uniform(-1.0, 1.0),
                        rng.uniform(0.8, 1.6)])
        sw.append(m)
        ws.append(inv)
    return np.stack(ws), np.stack(sw)


def timed(fn):
    a = time.perf_counter()
    fn()
    return (time.perf_counter() - a) * 1e3  # every call ends in a device synchronisation


def spread(ts):
    ts = sorted(ts)
    return {"median": ts[len(ts) // 2], "min": ts[0], "max": ts[-1], "runs": len(ts)}


def run_case(name, cfg, block_size, frames, rounds):
    p = synth.params(cfg)
    p.grid_opacity = 40
    if block_size is not None:
        p.block_size = block_size
    n = synth.points_per_frame(cfg)
    src = synth.frames(cfg, 0, 64)
    host = np.ascontiguousarray(np.concatenate([src] * (frames // 64 + 1))[:frames])
    dev = torch.from_numpy(host).to("cuda:0")
    counts = np.full(frames, n, np.int32)
    ws, sw = poses(p, frames)
    out = {"config": cfg, "block_size": float(p.block_size), "frames_per_call": frames, "points_per_frame": n,
           "input_bytes": int(host.nbytes)}
    with ObstacleProcessor(p, n, max_batch=frames) as op:
        W, H = op.occupancy_dims()
        out["grid"] = {"W": W, "H": H, "cells": W * H}
        g_dev = torch.empty((frames, H, W), dtype=torch.int8, device="cuda:0")
        g_pin = torch.empty((frames, H, W), dtype=torch.int8).pin_memory()
        a = lambda: op.process_batch_raw(dev.data_ptr(), n, counts)
        b = lambda: op.process_batch_occupancy_raw(dev.data_ptr(), n, counts, ws, sw, g_dev.data_ptr())
        c = lambda: op.process_batch_occupancy_raw(dev.data_ptr(), n, counts, ws, sw, g_pin.data_ptr())
        g_np = np.empty((frames, H, W), np.int8)
        c2 = lambda: op.process_batch_occupancy_raw(dev.data_ptr(), n, counts, ws, sw, g_np.ctypes.data)
        for fn in (a, b, c, c2, a, b, c, c2):  # warm-up: module loads, pinned result buffers, grid scratch
            fn()
        ta, tb, tc, tc2 = [], [], [], []
        for _ in range(rounds):
            ta.append(timed(a))
            tb.append(timed(b))
            tc.append(timed(c))
            tc2.append(timed(c2))
        out["a_process_batch_ms"] = spread(ta)
        out["b_batch_occupancy_grids_device_ms"] = spread(tb)
        out["c_batch_occupancy_grids_pinned_host_ms"] = spread(tc)
        out["c_pageable_batch_occupancy_grids_pageable_host_ms"] = spread(tc2)
        out["b_minus_a_us_per_frame"] = (out["b_batch_occupancy_grids_device_ms"]["median"] -
                                         out["a_process_batch_ms"]["median"]) * 1e3 / frames
        out["c_minus_a_us_per_frame"] = (out["c_batch_occupancy_grids_pinned_host_ms"]["median"] -
                                         out["a_process_batch_ms"]["median"]) * 1e3 / frames
        # per-kernel device time of the grid kernels (a call of its own: timing serialises the lanes)
        op.enable_kernel_timing(True)
        b()
        kt = op.kernel_times()
        op.enable_kernel_timing(False)
        out["grid_kernels_us_per_frame"] = {k: kt[k][0] / frames for k in GRID_KERNELS if k in kt}
        out["grid_kernel_launches"] = {k: kt[k][1] for k in GRID_KERNELS if k in kt}

        # d: today's chain, frames resident in HBM, results and grids on the host
        grid = np.empty((H, W), np.int8)
        lib, h = op._lib, op._h

        def chain():
            res = op.process_batch_raw(dev.data_ptr(), n, counts)
            for f in range(frames):
                r = res[f]
                op._check(lib.pcop_occupancy_grid(h, C.c_void_p(dev.data_ptr() + f * n * 16), n,
                                                  grid.ctypes.data_as(C.c_void_p), None, None))
                op._check(lib.pcop_occupancy_shadows(h, C.cast(r.remaining_cloud, C.c_void_p), r.n_remaining,
                                                     C.cast(r.cluster_offsets, C.c_void_p),
                                                     C.cast(r.cluster_indices, C.c_void_p), r.n_clusters,
                                                     ws[f].ctypes.data_as(C.c_void_p), sw[f].ctypes.data_as(C.c_void_p),
                                                     grid.ctypes.data_as(C.c_void_p), None, None))
        chain()
        td = [timed(chain) for _ in range(max(2, rounds // 3))]
        out["d_chain_ms"] = spread(td)
        out["d_minus_a_us_per_frame"] = (out["d_chain_ms"]["median"] - out["a_process_batch_ms"]["median"]) * 1e3 / frames
        ba = out["b_minus_a_us_per_frame"]
        out["grid_product_speedup_d_minus_a_over_b_minus_a"] = out["d_minus_a_us_per_frame"] / ba if ba > 0 else None
        out["call_speedup_d_over_b"] = out["d_chain_ms"]["median"] / out["b_batch_occupancy_grids_device_ms"]["median"]
        out["per_frame_us"] = {k: out[key]["median"] * 1e3 / frames for k, key in
                               (("a", "a_process_batch_ms"), ("b", "b_batch_occupancy_grids_device_ms"),
                                ("c", "c_batch_occupancy_grids_pinned_host_ms"),
                                ("c_pageable", "c_pageable_batch_occupancy_grids_pageable_host_ms"), ("d", "d_chain_ms"))}
    del dev, g_dev, g_pin
    torch.cuda.empty_cache()

    # single-frame latency, host frame in, host grid out
    with ObstacleProcessor(p, n, max_batch=1) as op:
        cloud = src[0]
        w1, s1 = ws[:1], sw[:1]

        def chain1():
            g0, _, _ = op.occupancy_grid(cloud)
            fr = op.process(cloud)
            op.handle_shadow_casting(g0, fr.remaining_cloud, fr.cluster_offsets, fr.cluster_indices, w1[0], s1[0])

        one = lambda: op.process_batch_occupancy(cloud[None], w1, s1)
        for _ in range(5):
            chain1()
            one()
        t1, t2 = [], []
        for _ in range(31):
            t1.append(timed(chain1))
            t2.append(timed(one))
        out["single_frame_p50_ms"] = {"three_call_chain": spread(t1)["median"], "batch_occupancy_batch1": spread(t2)["median"]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--round", default="r03")
    ap.add_argument("--out", default=None)
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("occupancy_batch_bench: no CUDA device (nothing is measured without one)")
    result = {"card": card(), "cases": {}}
    for name, cfg, bs in CASES:
        result["cases"][name] = run_case(name, cfg, bs, args.frames, args.rounds)
        print(name, json.dumps({k: v for k, v in result["cases"][name].items()
                                if k in ("per_frame_us", "b_minus_a_us_per_frame", "grid_product_speedup_d_minus_a_over_b_minus_a", "call_speedup_d_over_b",
                                         "single_frame_p50_ms", "grid_kernels_us_per_frame")}), flush=True)
    result["card_after"] = card()
    path = args.out or os.path.join(ROOT, "profiles", f"occupancy_batch_{args.round}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
