"""bench.py --dump-outputs on CPU: the writer gets oracle results in the library's result struct and must store every
frame's counts and plane records, and the result arrays of its frame sample, as float32 / float64 within the size cap."""
import ctypes as C
import os

import numpy as np

import bench
import oracle_lib as O
from pointcloud_obstacle_processing_b200 import Frame, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi


def _oracle_results(count):
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    res = (abi.FrameResult * count)()
    for k in range(count):
        cloud = synth.frame(1, k)
        assert O.lib().pcop_oracle_process(C.byref(p), cloud.ctypes.data_as(C.c_void_p), len(cloud), C.byref(res[k])) == 0
    return res


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_outputs_stores_every_result(tmp_path, monkeypatch):
    res = _oracle_results(3)
    try:
        frames = [Frame.from_c(r) for r in res]
        bench.dump_outputs(res, str(tmp_path / "all"))
        monkeypatch.setattr(bench, "DUMP_LIMIT", 700 << 10)  # room for the first frame's arrays only (~460 KB)
        bench.dump_outputs(res, str(tmp_path / "capped"))
    finally:
        for r in res:
            O.lib().pcop_oracle_free_result(C.byref(r))

    d = _load(tmp_path / "all")
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert d["frame_index"].tolist() == [0, 1, 2]
    for k in bench.SCALAR_FIELDS:
        assert d[k].tolist() == [getattr(f, k) for f in frames]
    for k, f in enumerate(frames):
        np.testing.assert_array_equal(d["plane_pass_points"][k, :f.n_plane_passes], f.plane_pass_points)
        np.testing.assert_array_equal(d["plane_pass_coeff"][k, :f.n_plane_passes], f.plane_pass_coeff)
        np.testing.assert_array_equal(d["plane_coeff"][k], f.plane_coeff)
    for name in bench.ARRAY_FIELDS:
        want = np.concatenate([getattr(f, name) for f in frames])
        assert d[name].dtype == (np.float32 if want.dtype == np.float32 else np.float64)
        np.testing.assert_array_equal(d[name], want)

    capped = tmp_path / "capped"
    assert sum(os.path.getsize(capped / f) for f in os.listdir(capped)) <= 700 << 10
    c = _load(capped)
    assert c["frame_index"].tolist() == [0]
    np.testing.assert_array_equal(c["remaining_cloud"], frames[0].remaining_cloud)
    np.testing.assert_array_equal(c["n_clusters"], d["n_clusters"])
