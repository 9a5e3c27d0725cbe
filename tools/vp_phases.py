"""Phase breakdown (clock64 of block (frame 5, group 20)) of the partition voxel path's reduce kernel, and the group
counts of one call: groups per frame, groups that take the binary search instead of the direct bucket table, groups of
more than 64 buckets, elements per group.
Needs a library built with PCOP_NVCC_EXTRA=-DPCOP_VP_DEBUG_CLK (python -m pointcloud_obstacle_processing_b200._build --force)."""
import ctypes as C
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth, load_library

NAMES = ["setup (bucket table, clears)", "pass 1 (load, key, bit)", "popcount round totals", "round bases + pass 2",
         "run lengths: round totals + look-back", "run lengths: starts", "pass 3a (indices by voxel)",
         "pass 3b (rank in run, stage xyz)", "sums + centroid stores"]
p = synth.params(2)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8
clouds = synth.frames(2, 0, B)
lib = load_library()
out = (C.c_longlong * 16)()
with ObstacleProcessor(p, clouds.shape[1], max_batch=B) as op:
    for _ in range(3):
        op.process_batch(clouds, np.full(B, clouds.shape[1], np.int32))
    assert lib.pcop_debug_vp_reduce_cycles(out) == 0  # (also clears the group counters)
    op.process_batch(clouds, np.full(B, clouds.shape[1], np.int32))
    st = lib.pcop_debug_vp_reduce_cycles(out)
    assert st == 0, st
t = list(out)
for k, name in enumerate(NAMES):
    print("%-38s %9d cycles" % (name, t[k + 1] - t[k]))
print("%-38s %9d cycles" % ("total", t[len(NAMES)] - t[0]))
groups, bsearch, wide, elems = t[12:16]
print("frames %d: %.2f groups per frame, %d on the binary search, %d of more than 64 buckets, %.0f elements per group"
      % (B, groups / B, bsearch, wide, elems / max(groups, 1)))
