"""Obstacle footprints (PCOP_OUT_FOOTPRINTS): what the box and hull kernels add to a call.

python tools/footprints_bench.py [--round r09] [--out PATH] [--rounds 7] [--ab-parent DIR]

Cases (one step = one call; off = outputs without the bit, on = with it; the two alternate within every round, median
and min .. max over the rounds):
  config2_b1024_host     bench config 2, 1024 frames per call, OUT_DEFAULT (| OUT_FOOTPRINTS), results to the host
  config2_b1024_device   the same with OUT_DEVICE: results left in HBM
  config3_single         bench config 3, one frame per call (p50 of the calls)
  config4_single         bench config 4, one frame per call (its 300 k-point blobs take the multi-piece path)
Per case also: the per-kernel device times of one call with kernel timing on, the footprint launches, and a check that
the on call's results equal the off call's and its footprints equal the C++ restatement (footprint_util).
--ab-parent DIR: a checkout of the parent build; runs bench.py --steps 10 --warmup 3 --no-configs from DIR and from
this tree, alternating, twice each.
Writes profiles/footprints_<round>.json (or --out)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # device memory for the frames only

import footprint_util as F
from occupancy_batch_bench import card, spread, timed
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi

CASES = [("config2_b1024_host", 2, 1024, False), ("config2_b1024_device", 2, 1024, True),
         ("config3_single", 3, 1, False), ("config4_single", 4, 1, False)]


def run_case(name, cfg, frames, device, rounds):
    p = synth.params(cfg)
    p.publish_point_clouds = 0
    n = synth.points_per_frame(cfg)
    src = synth.frames(cfg, 0, min(frames, 64))
    host = np.ascontiguousarray(np.concatenate([src] * (frames // len(src) + 1))[:frames])
    dev = torch.from_numpy(host).to("cuda:0")
    counts = np.full(frames, n, np.int32)
    masks = {"off": abi.OUT_DEFAULT, "on": abi.OUT_DEFAULT | abi.OUT_FOOTPRINTS}
    if device:
        masks = {k: v | abi.OUT_DEVICE for k, v in masks.items()}
    out = {"config": cfg, "frames_per_call": frames, "results_in_hbm": device}
    with ObstacleProcessor(p, n, max_batch=frames) as op:
        def call(mask):
            q = p.copy()
            q.outputs = mask
            op.set_params(q)
            return timed(lambda: op.process_batch_raw(dev.data_ptr(), n, counts))

        for _ in range(2):  # warm-up of both shapes
            for m in masks.values():
                call(m)
        ts = {k: [] for k in masks}
        for _ in range(rounds):
            for k, m in masks.items():
                ts[k].append(call(m))
        for k in masks:
            out[f"{k}_ms"] = spread(ts[k])
        out["on_over_off"] = out["on_ms"]["median"] / out["off_ms"]["median"]
        # per-kernel times (kernel timing serialises the lanes: a separate call, not the timed ones)
        op.enable_kernel_timing(True)
        call(masks["on"])
        kt = op.kernel_times()
        launches = op.last_launch_count
        op.enable_kernel_timing(False)
        call(masks["off"])
        out["launches_off"] = op.last_launch_count
        out["launches_on"] = launches
        out["footprint_kernels_us"] = {k: v[0] for k, v in kt.items() if k.startswith("k_fp_")}
        out["footprint_launches"] = {k: v[1] for k, v in kt.items() if k.startswith("k_fp_")}
        out["all_kernels_us_on"] = sum(v[0] for v in kt.values())
        # results: the on call equals the off call, and its footprints the C++ restatement (a few frames)
        if not device:
            q = p.copy()
            q.outputs = masks["off"]
            op.set_params(q)
            off = op.process_batch(host[:4])
            q.outputs = masks["on"]
            op.set_params(q)
            on = op.process_batch(host[:4])
            same = True
            hulls = []
            for a, b in zip(off, on):
                for k in ("remaining_cloud", "cluster_offsets", "cluster_indices", "obstacles"):
                    same = same and getattr(a, k).tobytes() == getattr(b, k).tobytes()
                ref = F.oracle_footprints(b.remaining_cloud, b.cluster_offsets, b.cluster_indices)
                same = same and all(x.tobytes() == y.tobytes() for x, y in zip((b.boxes, b.hull_offsets, b.hull_indices), ref))
                hulls.append([int(b.n_clusters), int(len(b.hull_indices)), int(np.diff(b.cluster_offsets).max(initial=0))])
            out["results_equal_and_footprints_exact"] = bool(same)
            out["clusters_hull_vertices_largest_cluster"] = hulls
    return out


def ab_parent(parent, rounds=2):
    """bench.py from the parent checkout and from this tree, alternating"""
    runs, parent = [], os.path.abspath(parent)
    for r in range(rounds):
        for tag, root in (("parent", parent), ("new", ROOT)):
            line = subprocess.check_output([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "10",
                                            "--warmup", "3", "--no-configs"], cwd=root).decode().strip().splitlines()[-1]
            runs.append({"build": tag, "round": r, "bench": json.loads(line)})
            print(tag, line, flush=True)
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--round", default="r09")
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--ab-parent", default=None, metavar="DIR")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("footprints_bench: no CUDA device (nothing is measured without one)")
    result = {"card": card(), "cases": {}}
    for name, cfg, frames, device in CASES:
        result["cases"][name] = run_case(name, cfg, frames, device, args.rounds)
        c = result["cases"][name]
        print(name, json.dumps({k: v for k, v in c.items() if k.endswith("_ms") or k.startswith(("on_", "footprint", "launches"))}),
              flush=True)
    if args.ab_parent:
        result["ab_parent"] = ab_parent(args.ab_parent)
    result["card_after"] = card()
    path = args.out or os.path.join(ROOT, "profiles", f"footprints_{args.round}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
