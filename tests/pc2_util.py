"""sensor_msgs/PointCloud2 payloads for the batched-ingest tests and benchmark: TEST INFRASTRUCTURE.

Packs float32 [n, 4] clouds into the record layouts real drivers produce, moves synthetic world frames into a seeded
sensor frame, and decodes messages the reference way (oracle fromPCLPointCloud2 + transformPointCloud)."""
import numpy as np

import oracle_lib as O
from shadow_util import rigid

# name: (point_step, off_x, off_y, off_z)
LAYOUTS = {
    "xyz16": (16, 0, 4, 8),      # pcl::toROSMsg(PointXYZ): x y z pad
    "xyzir32": (32, 0, 4, 8),    # Velodyne XYZIR: x y z pad, intensity float at 16, ring uint16 at 20, padding
    "xyzrgb32": (32, 0, 4, 8),   # Kinect XYZRGB: x y z pad, rgb at 16, padding
    "xyz22": (22, 0, 4, 8),      # packed records: every record after the first starts off a 4-byte boundary
    "zxy26": (26, 17, 21, 13),   # permuted, odd offsets: z x y at 13, 17, 21
}


def pack(cloud, layout, seed=0):
    """the PointCloud2.data bytes (uint8 [n * point_step]) of cloud[:, :3] in `layout`; the other bytes carry filler
    (intensity / ring / rgb for the 32-byte layouts, random bytes elsewhere)"""
    step, ox, oy, oz = LAYOUTS[layout]
    n = len(cloud)
    rng = np.random.default_rng(seed)
    rec = rng.integers(0, 256, size=(n, step), dtype=np.uint8)
    if layout == "xyzir32":
        rec[:, 16:20] = rng.uniform(0, 255, n).astype(np.float32).view(np.uint8).reshape(n, 4)
        rec[:, 20:22] = rng.integers(0, 64, n).astype(np.uint16).view(np.uint8).reshape(n, 2)
    elif layout == "xyzrgb32":
        rec[:, 16:20] = rng.integers(0, 1 << 24, n).astype(np.uint32).view(np.uint8).reshape(n, 4)
    for a, off in enumerate((ox, oy, oz)):
        rec[:, off:off + 4] = np.ascontiguousarray(cloud[:, a], np.float32).view(np.uint8).reshape(n, 4)
    return rec.reshape(-1)


def sensor_poses(p, B, seed):
    """one sensor pose per frame: (sensor_to_world [B, 4, 4], world_to_sensor [B, 4, 4])"""
    rng = np.random.default_rng(seed)
    sw, ws = [], []
    for _ in range(B):
        m, inv = rigid(rng.uniform(-0.3, 0.3), rng.uniform(0.3, 0.6), 0.0,
                       [p.x_max + rng.uniform(0.2, 1.5), 0.5 * (p.y_min + p.y_max) + rng.uniform(-1.0, 1.0),
                        rng.uniform(0.8, 1.6)])
        sw.append(m)
        ws.append(inv)
    return np.stack(sw), np.stack(ws)


def to_sensor(cloud, world_to_sensor):
    """a world-frame cloud as the sensor saw it (float32 [n, 4], padding 1)"""
    return O.transform(cloud, world_to_sensor, is_dense=True)


def decode(payload, n, layout, transform=None, is_dense=False):
    """the reference chain for one message: fromPCLPointCloud2<PointXYZ>, then transformPointCloud (None: none)"""
    step, ox, oy, oz = LAYOUTS[layout]
    n = int(n)
    xyz = O.pointcloud2_to_xyz(payload, n, step, ox, oy, oz) if n else np.zeros((0, 4), np.float32)
    return xyz if transform is None or n == 0 else O.transform(xyz, transform, is_dense=is_dense)


def decode_batch(payloads, counts, layouts, transforms=None, dense=None, cap=None):
    """decode() of every message into one [B, cap, 4] array (cap: the largest count) for pcop_process_batch"""
    B = len(payloads)
    cap = cap or max(1, max(counts))
    out = np.zeros((B, cap, 4), np.float32)
    for f in range(B):
        out[f, :counts[f]] = decode(payloads[f], counts[f], layouts[f], None if transforms is None else transforms[f],
                                    False if dense is None else dense[f])
    return out
