"""Accumulation windows: pcop_process_batch_pointcloud2_windows against pcop_process_batch on pre-decoded
concatenations and against the per-window accumulate chain it replaces.

python tools/pointcloud2_windows_bench.py [--round r07] [--out PATH] [--rounds 7] [--ab-parent DIR]

Cases (frames of K posed sensor-frame messages each; 64 distinct messages and poses tiled, payloads and clouds resident
in HBM, larger than the 126 MB L2; one step = one call):
  config1_k2_xyzrgb32    config-1 messages as 32-byte XYZRGB, K = 2 (the node's code default), 512 frames
  config2_rig_xyzir32    two HDL-64 sensors (config-2 messages, 32-byte XYZIR) per time step, 256 frames
  config1_k20_xyzrgb32   config-1 messages, K = 20: 600 000-point frames (the LSD voxel path), 32 frames
and per case:
  a   pcop_process_batch on the concatenations the oracle decodes from the same messages
  b   the windows call, device payloads
  c   the windows call, pinned host payloads
  d   the per-window chain pcop_accumulate_reset + K pcop_accumulate_pointcloud2 + pcop_process_accumulated
a, b and c alternate within every round (the spread is the min .. max over rounds); d runs fewer rounds.  Every frame
count of b equals a's (checked after the timed rounds).  The decode kernel's device time comes from a separate call with
kernel timing on; its rate is (point_step + 16) bytes per record.  The host time of classifying the payload pointers, one
cudaPointerGetAttributes per message against one driver query per allocation, comes from tools/ubench/payload_classify.cu
(built into a temporary directory) on each case's message count and payload size.
--ab-parent DIR: a checkout of the parent build; runs tools/pointcloud2_batch_bench.py (the one-message cases) and
bench.py --steps 10 --warmup 3 --no-configs from DIR and from this tree, alternating, twice each.
Writes profiles/pointcloud2_windows_<round>.json (or --out)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

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

CASES = [("config1_k2_xyzrgb32", 1, "xyzrgb32", 2, 512), ("config2_rig_xyzir32", 2, "xyzir32", 2, 256),
         ("config1_k20_xyzrgb32", 1, "xyzrgb32", 20, 32)]


def classify_us(messages, bytes_per_message):
    """tools/ubench/payload_classify.cu on this card: host us per call, per message vs per allocation"""
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "payload_classify")
        subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a",
                               "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tools", "ubench", "payload_classify.cu"),
                               "-o", exe, "-lcudart"])
        return json.loads(subprocess.check_output([exe, str(messages), str(bytes_per_message)]).decode())


def run_case(name, cfg, layout, K, frames, rounds):
    p = synth.params(cfg)
    n1 = synth.points_per_frame(cfg)
    step = LAYOUTS[layout][0]
    M = frames * K
    cap = K * n1
    D = 64
    world = synth.frames(cfg, 0, D)
    sw_d, ws_d = sensor_poses(p, D, 1)
    payload_d = np.stack([pack(to_sensor(world[k], ws_d[k]), layout, k) for k in range(D)])  # [D, n1 * step]
    decoded_d = torch.from_numpy(np.stack([decode(payload_d[k], n1, layout, sw_d[k]) for k in range(D)])).to("cuda:0")
    tile = np.arange(M) % D  # message m = distinct message m % D
    sw = np.ascontiguousarray(sw_d[tile])
    idx = torch.from_numpy(tile).to("cuda:0")
    dev_payload = torch.from_numpy(payload_d).to("cuda:0").index_select(0, idx).contiguous()
    pin_payload = torch.empty((M, n1 * step), dtype=torch.uint8).pin_memory()
    for m in range(M):
        pin_payload[m].copy_(torch.from_numpy(payload_d[tile[m]]))
    concat = decoded_d.index_select(0, idx).reshape(frames, cap, 4).contiguous()  # the frames a pre-decoding caller has
    del decoded_d
    counts = np.full(frames, cap, np.int32)
    first = (np.arange(frames + 1) * K).astype(np.int32)
    out = {"config": cfg, "layout": layout, "point_step": step, "messages_per_frame": K, "frames_per_call": frames,
           "messages_per_call": M, "points_per_message": n1, "points_per_frame": cap,
           "payload_bytes": int(M * n1 * step), "decoded_cloud_bytes": int(concat.numel() * 4)}

    def descs(base):
        arr = (abi.PointCloud2Frame * M)()
        for m in range(M):
            arr[m] = abi.PointCloud2Frame(base + m * n1 * step, n1, *LAYOUTS[layout], 0)
        return arr
    d_dev, d_pin = descs(dev_payload.data_ptr()), descs(pin_payload.data_ptr())
    t16 = sw.reshape(-1, 16).ctypes.data_as(C.c_void_p)
    fp = first.ctypes.data_as(C.c_void_p)
    with ObstacleProcessor(p, cap, max_batch=frames) as op:
        lib, h = op._lib, op._h
        res = (abi.FrameResult * frames)()

        def win(arr):
            op._check(lib.pcop_process_batch_pointcloud2_windows(h, arr, M, fp, frames, t16, None, None, None, res))
        a = lambda: op.process_batch_raw(concat.data_ptr(), cap, counts)
        b = lambda: win(d_dev)
        c = lambda: win(d_pin)
        for fn in (a, b, c, a, b, c):  # warm-up: module loads, pinned result buffers, staging, descriptors
            fn()
        ta, tb, tc = [], [], []
        for _ in range(rounds):
            ta.append(timed(a))
            tb.append(timed(b))
            tc.append(timed(c))
        b()
        key = lambda r: (r.n_input, r.n_crop, r.n_voxel, r.n_sor, r.n_remaining, r.n_clusters, r.n_cluster_points, r.warnings)
        got = [key(r) for r in res]
        out["b_counts_equal_a"] = got == [key(r) for r in a()]
        out["a_process_batch_ms"] = spread(ta)
        out["b_windows_device_payloads_ms"] = spread(tb)
        out["c_windows_pinned_host_payloads_ms"] = spread(tc)
        med = lambda k: out[k]["median"] * 1e3
        out["b_minus_a_us"] = {"per_message": (med("b_windows_device_payloads_ms") - med("a_process_batch_ms")) / M,
                               "per_frame": (med("b_windows_device_payloads_ms") - med("a_process_batch_ms")) / frames}
        out["c_minus_a_us_per_message"] = (med("c_windows_pinned_host_payloads_ms") - med("a_process_batch_ms")) / M
        out["c_upload_GBps_if_bound_by_the_payload_copy"] = M * n1 * step / (out["c_windows_pinned_host_payloads_ms"]["median"] * 1e6)

        op.enable_kernel_timing(True)  # the decode kernel alone (a call of its own: timing serialises the lanes)
        b()
        us, launches = op.kernel_times()["k_pc2_ingest"]
        op.enable_kernel_timing(False)
        out["decode_kernel"] = {"us_per_message": us / M, "launches": launches, "GBps": (step + 16) * n1 * M / (us * 1e3)}

        one = abi.FrameResult()

        def chain():
            for f in range(frames):
                op._check(lib.pcop_accumulate_reset(h))
                for m in range(f * K, (f + 1) * K):
                    op._check(lib.pcop_accumulate_pointcloud2(h, C.c_void_p(d_dev[m].data), n1, *LAYOUTS[layout],
                                                              sw[m].ctypes.data_as(C.c_void_p), 0, None))
                op._check(lib.pcop_process_accumulated(h, C.byref(one)))
        chain()
        td = [timed(chain) for _ in range(max(2, rounds // 3))]
        out["d_chain_ms"] = spread(td)
        out["d_over_b"] = out["d_chain_ms"]["median"] / out["b_windows_device_payloads_ms"]["median"]
    out["classify_host_us_per_call"] = classify_us(M, n1 * step)
    del dev_payload, pin_payload, concat
    torch.cuda.empty_cache()
    return out


def ab_parent(parent, rounds=2):
    """the one-message cases and bench.py from the parent checkout and from this tree, alternating"""
    runs = []
    with tempfile.TemporaryDirectory() as d:
        for r in range(rounds):
            for tag, root in (("parent", parent), ("new", ROOT)):
                path = os.path.join(d, f"{tag}{r}.json")
                subprocess.check_call([sys.executable, os.path.join(root, "tools", "pointcloud2_batch_bench.py"), "--out", path],
                                      stdout=subprocess.DEVNULL)
                cases = json.load(open(path))["cases"]
                line = subprocess.check_output([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "10",
                                                "--warmup", "3", "--no-configs"], cwd=root).decode().strip().splitlines()[-1]
                runs.append({"build": tag, "round": r,
                             "pointcloud2_batch": {k: {"per_frame_us": v["per_frame_us"], "decode_kernel": v["decode_kernel"],
                                                       "b_counts_equal_a": v["b_counts_equal_a"]} for k, v in cases.items()},
                             "bench": json.loads(line)})
                print(json.dumps(runs[-1]["pointcloud2_batch"]), line, flush=True)
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--round", default="r07")
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--ab-parent", default=None, metavar="DIR")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pointcloud2_windows_bench: no CUDA device (nothing is measured without one)")
    result = {"card": card(), "cases": {}}
    for name, cfg, layout, K, frames in CASES:
        result["cases"][name] = run_case(name, cfg, layout, K, frames, args.rounds)
        print(name, json.dumps({k: v for k, v in result["cases"][name].items()
                                if k in ("b_minus_a_us", "decode_kernel", "b_counts_equal_a", "d_over_b",
                                         "classify_host_us_per_call")}), flush=True)
    if args.ab_parent:
        result["ab_parent"] = ab_parent(args.ab_parent)
    result["card_after"] = card()
    path = args.out or os.path.join(ROOT, "profiles", f"pointcloud2_windows_{args.round}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
