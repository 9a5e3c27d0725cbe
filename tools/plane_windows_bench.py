"""Plane-stage timing of one build, and an output digest per case to compare builds.

    python tools/plane_windows_bench.py --out a.json [--reps 20]        # the package of this tree
    python tools/plane_windows_bench.py --compare a.json b.json ...     # digests equal? medians side by side

Per case: the device time of the plane kernels per call (every kernel named k_plane*, kernel timing on) and the wall
time of a whole call with kernel timing off (host frames in, results on the host; the synthetic cases run the plane
stage alone, the synth-config cases the whole pipeline).  Cases:
  hdl64_256     256 BASELINE configs[1] frames (plane inputs of about 55 000 points: small tier)
  cfg2_2cm_64   64 configs[1] frames at a 2 cm voxel leaf (about 100 000 points: the large tier in one window)
  cfg3_16       the 16 BASELINE configs[2] frames bench.py runs (128 353 .. 134 047 points)
  plane_<n>_b<B> B synthetic plane inputs of n points (crop, voxel, SOR and clustering off)
The digest hashes every field of every frame of the last call."""
import argparse
import dataclasses
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def planes_cloud(rng, n, fracs, noise=0.01):
    """planes of decreasing size plus uniform clutter (tests/test_gpu_parity.py): one pass per plane"""
    parts = []
    for k, fr in enumerate(fracs):
        m = int(n * fr)
        uv = rng.uniform(-20, 20, size=(m, 2))
        nrm = rng.normal(size=3)
        nrm /= np.linalg.norm(nrm)
        e1 = np.cross(nrm, [1.0, 0.3, 0.2])
        e1 /= np.linalg.norm(e1)
        e2 = np.cross(nrm, e1)
        parts.append(uv[:, :1] * e1 + uv[:, 1:] * e2 + nrm * (3.0 * k) + rng.normal(size=(m, 1)) * noise * nrm)
    parts.append(rng.uniform(-25, 25, size=(n - sum(len(q) for q in parts), 3)))
    pts = np.concatenate(parts).astype(np.float32)[rng.permutation(n)]
    return np.concatenate([pts, np.ones((n, 1), np.float32)], axis=1)


def cases(synth):
    out = []
    out.append(("hdl64_256", synth.params(2), synth.frames(2, 0, 256)))
    p = synth.params(2)
    p.downsample_size = 0.02
    out.append(("cfg2_2cm_64", p, synth.frames(2, 0, 64)))
    out.append(("cfg3_16", synth.params(3), synth.frames(3, 0, 16)))
    for n, B in ((150000, 1), (150000, 16), (300000, 1), (300000, 16), (1000000, 1), (1000000, 8)):
        p = synth.params(2)
        p.enable_crop = p.enable_voxel = p.enable_sor = p.enable_cluster = 0
        rng = np.random.default_rng(n + B)
        out.append((f"plane_{n}_b{B}", p, np.stack([planes_cloud(rng, n, (0.4, 0.2, 0.15)) for _ in range(B)])))
    return out


def digest(frames):
    h = hashlib.sha256()
    for fr in frames:
        for f in dataclasses.fields(fr):
            v = getattr(fr, f.name)
            h.update(f.name.encode())
            h.update(np.ascontiguousarray(v).tobytes() if isinstance(v, np.ndarray) else repr(v).encode())
    return h.hexdigest()


def measure(reps):
    sys.path.insert(0, ROOT)
    from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
    from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi
    res = {}
    for name, p, clouds in cases(synth):
        p.outputs = abi.OUT_ALL
        B, n = clouds.shape[0], clouds.shape[1]
        with ObstacleProcessor(p, n, max_batch=B) as op:
            for _ in range(3):  # warm-up; also settles the lane's route history
                frames = op.process_batch(clouds)
            op.enable_kernel_timing(True)
            for _ in range(reps):
                op.process_batch(clouds)
            kt = op.kernel_times()
            op.enable_kernel_timing(False)
            plane_us = sum(us for k, (us, _) in kt.items() if k.startswith("k_plane")) / reps
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter()
                frames = op.process_batch(clouds)
                ts.append((time.perf_counter() - t0) * 1e3)
        res[name] = {"frames": B, "points": n, "plane_kernel_us_per_call": plane_us,
                     "plane_kernels": sorted(k for k in kt if k.startswith("k_plane")),
                     "call_ms_median": float(np.median(ts)), "call_ms_min": float(np.min(ts)),
                     "call_ms_max": float(np.max(ts)), "plane_passes": [fr.n_plane_passes for fr in frames[:4]],
                     "digest": digest(frames)}
        print(name, json.dumps(res[name]), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--compare", nargs="+")
    a = ap.parse_args()
    if a.compare:
        runs = [(f, json.load(open(f))) for f in a.compare]
        for case in runs[0][1]["cases"]:
            ds = {r["cases"][case]["digest"] for _, r in runs}
            print(f"{case:22s} outputs {'equal' if len(ds) == 1 else 'DIFFER'}  " + "  ".join(
                f"{os.path.basename(f)}: {r['cases'][case]['plane_kernel_us_per_call']:9.1f} us "
                f"{r['cases'][case]['call_ms_median']:8.3f} ms" for f, r in runs))
        return
    import torch
    gpu = {"name": torch.cuda.get_device_name(0)}
    try:
        import subprocess
        gpu["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                                            capture_output=True, text=True).stdout.strip()
    except OSError:
        pass
    out = {"gpu": gpu, "reps": a.reps, "cases": measure(a.reps)}
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
