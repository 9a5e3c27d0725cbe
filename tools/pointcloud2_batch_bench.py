"""Batched PointCloud2 ingest: pcop_process_batch_pointcloud2 against pcop_process_batch on pre-decoded world clouds and
against the per-message chain it replaces.

python tools/pointcloud2_batch_bench.py [--round r04] [--out PATH] [--frames 1024] [--rounds 7]

Per case (config 2 HDL-64 frames as 32-byte XYZIR messages, config 1 frames as 32-byte XYZRGB messages, config 2 as a
packed 22-byte layout that takes the any-alignment decode), 1024 sensor-frame messages per call, each with its own pose
(64 distinct frames and poses tiled), payloads and clouds resident in HBM (larger than the 126 MB L2), one step = one
call:
  a       pcop_process_batch on the world clouds the oracle decodes from the same messages
  b       pcop_process_batch_pointcloud2, device payloads
  c       pcop_process_batch_pointcloud2, pinned host payloads
  b_grid  b with grids != NULL (grids into device memory)
  d       the per-message chain pcop_accumulate_reset + pcop_accumulate_pointcloud2 + pcop_process_accumulated
a, b, c and b_grid alternate within every round (the spread is the min .. max over rounds); d is slower by orders of
magnitude and runs fewer rounds.  Every frame count of b equals a's (checked after the timed rounds).  The decode kernel's
device time comes from a separate call with kernel timing on (which serialises the lanes); its achieved bandwidth is
(point_step + 16) bytes per record over that time, against the 6 544 GB/s a device-to-device copy reached on the same
card (DESIGN.md section 4).  The host time of classifying the payload pointers (one cudaPointerGetAttributes per message)
is timed with the same runtime call.  Writes profiles/pointcloud2_batch_<round>.json (or --out)."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # device and pinned memory for the resident payloads only

from occupancy_batch_bench import card, spread, timed
from pc2_util import LAYOUTS, decode, pack, sensor_poses, to_sensor
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi

CASES = [("config2_hdl64_xyzir32", 2, "xyzir32", 0.25), ("config1_xyzrgb32", 1, "xyzrgb32", None),
         ("config2_packed22", 2, "xyz22", 0.25)]
COPY_GBPS = 6544.3  # measured copy bandwidth of one B200 (DESIGN.md section 4)


def classify_us(ptrs):
    """host microseconds of one cudaPointerGetAttributes per pointer (what the call does per message)"""
    rt = None
    for name in ("libcudart.so.12", "libcudart.so"):
        try:
            rt = C.CDLL(name)
            break
        except OSError:
            continue
    if rt is None:
        return None
    attr = (C.c_char * 64)()
    rt.cudaPointerGetAttributes.argtypes = [C.c_void_p, C.c_void_p]
    for p in ptrs[:8]:
        rt.cudaPointerGetAttributes(attr, C.c_void_p(p))
    ts = []
    for _ in range(5):
        a = time.perf_counter()
        for p in ptrs:
            rt.cudaPointerGetAttributes(attr, C.c_void_p(p))
        ts.append((time.perf_counter() - a) * 1e6)
    return spread(ts)


def run_case(name, cfg, layout, block_size, frames, rounds):
    p = synth.params(cfg)
    p.grid_opacity = 40
    if block_size is not None:
        p.block_size = block_size
    n = synth.points_per_frame(cfg)
    step = LAYOUTS[layout][0]
    D = 64
    world = synth.frames(cfg, 0, D)
    sw_d, ws_d = sensor_poses(p, D, 1)
    payload_d = np.stack([pack(to_sensor(world[k], ws_d[k]), layout, k) for k in range(D)])  # [D, n * step]
    clouds_d = np.stack([decode(payload_d[k], n, layout, sw_d[k]) for k in range(D)])
    tile = np.arange(frames) % D
    sw, ws = np.ascontiguousarray(sw_d[tile]), np.ascontiguousarray(ws_d[tile])
    idx = torch.from_numpy(tile).to("cuda:0")
    dev_payload = torch.from_numpy(payload_d).to("cuda:0").index_select(0, idx).contiguous()
    pin_payload = torch.empty((frames, n * step), dtype=torch.uint8).pin_memory()
    for f in range(frames):
        pin_payload[f].copy_(torch.from_numpy(payload_d[tile[f]]))
    dev_clouds = torch.from_numpy(clouds_d).to("cuda:0").index_select(0, idx).contiguous()
    counts = np.full(frames, n, np.int32)
    out = {"config": cfg, "layout": layout, "point_step": step, "frames_per_call": frames, "points_per_frame": n,
           "payload_bytes": int(frames * n * step), "decoded_cloud_bytes": int(dev_clouds.numel() * 4)}

    def descs(base):
        arr = (abi.PointCloud2Frame * frames)()
        for f in range(frames):
            arr[f] = abi.PointCloud2Frame(base + f * n * step, n, *LAYOUTS[layout], 0)
        return arr
    d_dev, d_pin = descs(dev_payload.data_ptr()), descs(pin_payload.data_ptr())
    t16 = sw.reshape(-1, 16).ctypes.data_as(C.c_void_p)
    ws16 = ws.reshape(-1, 16).ctypes.data_as(C.c_void_p)
    with ObstacleProcessor(p, n, max_batch=frames) as op:
        W, H = op.occupancy_dims()
        g_dev = torch.empty((frames, H, W), dtype=torch.int8, device="cuda:0")
        lib, h = op._lib, op._h
        res = (abi.FrameResult * frames)()

        def pc2(arr, grids=None):
            op._check(lib.pcop_process_batch_pointcloud2(h, arr, frames, t16, ws16 if grids else None,
                                                         t16 if grids else None, C.c_void_p(grids) if grids else None, res))
        a = lambda: op.process_batch_raw(dev_clouds.data_ptr(), n, counts)
        b = lambda: pc2(d_dev)
        c = lambda: pc2(d_pin)
        bg = lambda: pc2(d_dev, g_dev.data_ptr())
        for fn in (a, b, c, bg, a, b, c, bg):  # warm-up: module loads, pinned result buffers, staging, grid scratch
            fn()
        ta, tb, tc, tg = [], [], [], []
        for _ in range(rounds):
            ta.append(timed(a))
            tb.append(timed(b))
            tc.append(timed(c))
            tg.append(timed(bg))
        b()
        got = [(r.n_input, r.n_crop, r.n_voxel, r.n_sor, r.n_remaining, r.n_clusters, r.n_cluster_points, r.warnings) for r in res]
        want = [(r.n_input, r.n_crop, r.n_voxel, r.n_sor, r.n_remaining, r.n_clusters, r.n_cluster_points, r.warnings)
                for r in op.process_batch_raw(dev_clouds.data_ptr(), n, counts)]
        out["b_counts_equal_a"] = got == want
        b()
        su = op.stage_times_us()
        out["b_stage_us_per_frame"] = {k: v / frames for k, v in su.items()}
        out["a_process_batch_ms"] = spread(ta)
        out["b_pc2_device_payloads_ms"] = spread(tb)
        out["c_pc2_pinned_host_payloads_ms"] = spread(tc)
        out["b_grid_pc2_device_payloads_grids_device_ms"] = spread(tg)
        med = lambda k: out[k]["median"] * 1e3 / frames
        out["per_frame_us"] = {"a": med("a_process_batch_ms"), "b": med("b_pc2_device_payloads_ms"),
                               "c": med("c_pc2_pinned_host_payloads_ms"),
                               "b_grid": med("b_grid_pc2_device_payloads_grids_device_ms")}
        out["b_minus_a_us_per_frame"] = out["per_frame_us"]["b"] - out["per_frame_us"]["a"]
        out["c_minus_a_us_per_frame"] = out["per_frame_us"]["c"] - out["per_frame_us"]["a"]
        out["c_upload_GBps_if_bound_by_the_payload_copy"] = frames * n * step / (out["c_pc2_pinned_host_payloads_ms"]["median"] * 1e6)

        # the decode kernel alone (a call of its own: timing serialises the lanes)
        op.enable_kernel_timing(True)
        b()
        kt = op.kernel_times()
        op.enable_kernel_timing(False)
        us, launches = kt["k_pc2_ingest"]
        out["decode_kernel"] = {"us_per_frame": us / frames, "launches": launches,
                                "GBps": (step + 16) * n * frames / (us * 1e3),
                                "share_of_copy_bandwidth": (step + 16) * n * frames / (us * 1e3) / COPY_GBPS}

        # d: the per-message chain, device payloads
        one = abi.FrameResult()

        def chain():
            for f in range(frames):
                op._check(lib.pcop_accumulate_reset(h))
                op._check(lib.pcop_accumulate_pointcloud2(h, C.c_void_p(d_dev[f].data), n, *LAYOUTS[layout],
                                                          sw[f].ctypes.data_as(C.c_void_p), 0, None))
                op._check(lib.pcop_process_accumulated(h, C.byref(one)))
        chain()
        td = [timed(chain) for _ in range(max(2, rounds // 3))]
        out["d_chain_ms"] = spread(td)
        out["per_frame_us"]["d"] = med("d_chain_ms")
        out["call_speedup_d_over_b"] = out["d_chain_ms"]["median"] / out["b_pc2_device_payloads_ms"]["median"]
        out["classify_host_us_per_call"] = {"device_payloads": classify_us([d_dev[f].data for f in range(frames)]),
                                            "pinned_payloads": classify_us([d_pin[f].data for f in range(frames)])}
    del dev_payload, pin_payload, dev_clouds, g_dev
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--round", default="r04")
    ap.add_argument("--out", default=None)
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pointcloud2_batch_bench: no CUDA device (nothing is measured without one)")
    result = {"card": card(), "cases": {}}
    for name, cfg, layout, bs in CASES:
        result["cases"][name] = run_case(name, cfg, layout, bs, args.frames, args.rounds)
        print(name, json.dumps({k: v for k, v in result["cases"][name].items()
                                if k in ("per_frame_us", "b_minus_a_us_per_frame", "c_minus_a_us_per_frame", "decode_kernel",
                                         "b_counts_equal_a", "call_speedup_d_over_b", "classify_host_us_per_call")}), flush=True)
    result["card_after"] = card()
    path = args.out or os.path.join(ROOT, "profiles", f"pointcloud2_batch_{args.round}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
