"""Depth-image ingest: pcop_process_batch_depth_windows against pcop_process_batch_pointcloud2_windows on the XYZRGB
messages depth_image_proc builds from the same images.

python tools/depth_windows_bench.py [--round r08] [--out PATH] [--rounds 7] [--ab-parent DIR]

Cases (16UC1 images of the config-3 scene, 32 distinct images and poses tiled, one pose per image; one step = one call):
  config3_16uc1_k1    640 x 480, windows of 1 image (a replay of single images), 256 frames
  config3_16uc1_k2    640 x 480, windows of 2 images, 128 frames
  qhd_16uc1_k2        960 x 540 (kinect2 qhd), windows of 2 images, 64 frames
and per case, on the same frames:
  a_dev / a_pin   pcop_process_batch_pointcloud2_windows on the point_step-32 XYZRGB payloads (depth_util.to_pointcloud2),
                  in HBM / in pinned host memory
  b_dev / b_pin   pcop_process_batch_depth_windows on the 16UC1 images, in HBM / in pinned host memory
The four alternate within every round (median and min .. max over the rounds).  Every result of b equals a's (counts,
plane records and warnings, checked after the timed rounds).  The decode kernels' device times come from one call of
each with kernel timing on; their rates count (bytes per input record + 16) per point, against the 6 544 GB/s copy
bandwidth of DESIGN §4.
--ab-parent DIR: a checkout of the parent build; runs bench.py --steps 10 --warmup 3 --no-configs from DIR and from
this tree, alternating, twice each.
Writes profiles/depth_windows_<round>.json (or --out)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # device and pinned memory for the payloads only

import depth_util as D
from occupancy_batch_bench import card, spread, timed
from pc2_util import LAYOUTS
from shadow_util import rigid
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi

COPY_GBPS = 6544.3  # device-to-device copy bandwidth of one B200 (DESIGN §4)
CASES = [("config3_16uc1_k1", D.CONFIG3, 1, 256), ("config3_16uc1_k2", D.CONFIG3, 2, 128), ("qhd_16uc1_k2", D.QHD, 2, 64)]


def run_case(name, camera, K, frames, rounds):
    p = synth.params(3)
    W, H, fx, fy, cx, cy = camera
    n1 = W * H
    M, Dn = frames * K, 32
    cap = K * n1
    rng = np.random.default_rng(1)
    images = [D.scene_image(k, camera) for k in range(Dn)]
    poses = np.stack([rigid(rng.uniform(-0.3, 0.3), rng.uniform(-0.1, 0.1), 0.0, rng.uniform(-0.4, 0.4, 3))[0]
                      for _ in range(Dn)]).astype(np.float32)
    depth_d = np.stack([np.ascontiguousarray(D.raw_bytes(im)) for im in images])  # [Dn, H * step]
    pc2_d = np.stack([D.to_pointcloud2(im, k) for k, im in enumerate(images)])   # [Dn, n1 * 32]
    tile = np.arange(M) % Dn
    idx = torch.from_numpy(tile).to("cuda:0")
    t16 = np.ascontiguousarray(poses[tile]).reshape(-1, 16)

    def resident(host):
        dev = torch.from_numpy(host).to("cuda:0").index_select(0, idx).contiguous()
        pin = torch.empty((M, host.shape[1]), dtype=torch.uint8).pin_memory()
        for m in range(M):
            pin[m].copy_(torch.from_numpy(host[tile[m]]))
        return dev, pin
    depth_dev, depth_pin = resident(depth_d)
    pc2_dev, pc2_pin = resident(pc2_d)
    first = (np.arange(frames + 1) * K).astype(np.int32)
    step = images[0].step

    def depth_descs(base):
        arr = (abi.DepthImageC * M)()
        for m in range(M):
            arr[m] = abi.DepthImageC(base + m * H * step, W, H, step, abi.DEPTH_16UC1, fx, fy, cx, cy)
        return arr

    def pc2_descs(base):
        arr = (abi.PointCloud2Frame * M)()
        for m in range(M):
            arr[m] = abi.PointCloud2Frame(base + m * n1 * 32, n1, *LAYOUTS["xyzrgb32"], 0)
        return arr
    dd, dp = depth_descs(depth_dev.data_ptr()), depth_descs(depth_pin.data_ptr())
    pd, pp = pc2_descs(pc2_dev.data_ptr()), pc2_descs(pc2_pin.data_ptr())
    tp, fp = t16.ctypes.data_as(C.c_void_p), first.ctypes.data_as(C.c_void_p)
    out = {"camera": {"width": W, "height": H, "fx": fx, "fy": fy, "cx": cx, "cy": cy}, "encoding": "16UC1",
           "images_per_frame": K, "frames_per_call": frames, "images_per_call": M, "points_per_frame": cap,
           "depth_payload_bytes": int(M * H * step), "pointcloud2_payload_bytes": int(M * n1 * 32)}
    with ObstacleProcessor(p, cap, max_batch=frames) as op:
        lib, h = op._lib, op._h
        res = (abi.FrameResult * frames)()
        key = lambda: [(r.n_input, r.n_crop, r.n_voxel, r.n_sor, r.n_remaining, r.n_clusters, r.n_cluster_points,
                        r.n_plane_passes, r.n_plane_inliers, tuple(r.plane_coeff), r.warnings) for r in res]

        def a(arr):
            return lambda: op._check(lib.pcop_process_batch_pointcloud2_windows(h, arr, M, fp, frames, tp, None, None,
                                                                                None, res))

        def b(arr):
            return lambda: op._check(lib.pcop_process_batch_depth_windows(h, arr, M, fp, frames, tp, None, None, None,
                                                                          res))
        fns = {"a_pointcloud2_device_ms": a(pd), "a_pointcloud2_pinned_ms": a(pp), "b_depth_device_ms": b(dd),
               "b_depth_pinned_ms": b(dp)}
        for _ in range(2):  # warm-up: module loads, pinned result buffers, staging, descriptors
            for fn in fns.values():
                fn()
        times = {k: [] for k in fns}
        for _ in range(rounds):
            for k, fn in fns.items():
                times[k].append(timed(fn))
        results = {}
        for k, fn in fns.items():
            fn()
            results[k] = key()
        out["b_results_equal_a"] = all(results[k] == results["a_pointcloud2_device_ms"] for k in results)
        for k in fns:
            out[k] = spread(times[k])
        med = lambda k: out[k]["median"]
        out["pinned_over_device"] = {"pointcloud2": med("a_pointcloud2_pinned_ms") / med("a_pointcloud2_device_ms"),
                                     "depth": med("b_depth_pinned_ms") / med("b_depth_device_ms")}
        out["b_minus_a_ms"] = {"device": med("b_depth_device_ms") - med("a_pointcloud2_device_ms"),
                               "pinned": med("b_depth_pinned_ms") - med("a_pointcloud2_pinned_ms")}
        for k, kernel, bpp in (("b_depth_device_ms", "k_depth_ingest", 2), ("a_pointcloud2_device_ms", "k_pc2_ingest", 32)):
            op.enable_kernel_timing(True)  # (a call of its own: timing serialises the lanes)
            fns[k]()
            us, launches = op.kernel_times()[kernel]
            op.enable_kernel_timing(False)
            gbps = (bpp + 16) * n1 * M / (us * 1e3)
            out["decode_kernel_" + kernel] = {"us_per_image": us / M, "launches": launches, "GBps": gbps,
                                              "share_of_copy_bandwidth": gbps / COPY_GBPS}
    del depth_dev, depth_pin, pc2_dev, pc2_pin
    torch.cuda.empty_cache()
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
    ap.add_argument("--round", default="r08")
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--ab-parent", default=None, metavar="DIR")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("depth_windows_bench: no CUDA device (nothing is measured without one)")
    result = {"card": card(), "cases": {}}
    for name, camera, K, frames in CASES:
        result["cases"][name] = run_case(name, camera, K, frames, args.rounds)
        c = result["cases"][name]
        print(name, json.dumps({k: v for k, v in c.items() if k.endswith("_ms") or k.startswith(("decode", "b_"))}),
              flush=True)
    if args.ab_parent:
        result["ab_parent"] = ab_parent(args.ab_parent)
    result["card_after"] = card()
    path = args.out or os.path.join(ROOT, "profiles", f"depth_windows_{args.round}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
