"""bench.py --dump-outputs: what it writes is float, bounded in size and the same sample on every run."""
import os

import numpy as np

import bench
from lld_slam_b200 import api, synth


def _read(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_keeps_small_results_whole(tmp_path):
    p = synth.make_local_ba_batch(2, 4, 50, 10, 3)
    out = api._ba_outputs(p, 22)
    out["pt_obs_bad"][::3] = 1
    out["trials_log"][:] = 7
    bench.dump_outputs(str(tmp_path), out)
    got = _read(tmp_path)
    assert sorted(got) == sorted(k for k, v in out.items() if isinstance(v, np.ndarray))
    for k, v in got.items():
        assert v.dtype in (np.float32, np.float64), k
        assert np.array_equal(v, out[k]), k


def test_dump_samples_large_results_to_a_fixed_subset(tmp_path):
    n = 5_000_000
    out = {"pt_xyz": np.arange(3 * n, dtype=np.float64).reshape(n, 3), "pt_obs_bad": (np.arange(n) % 2).astype(np.uint8),
           "n_iter_done": np.arange(8, dtype=np.int32).reshape(4, 2), "log_stride": 22}
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), out)
    bench.dump_outputs(str(b), out)
    total = sum(os.path.getsize(a / f) for f in os.listdir(a))
    assert total <= 64 * 10 ** 6
    ga, gb = _read(a), _read(b)
    for k in ga:
        assert np.array_equal(ga[k], gb[k]), k
    rows = ga["pt_xyz"][:, 0] / 3
    assert 0 < len(rows) < n and np.all(np.diff(rows) > 0)          # a subset of the rows, in order
    assert np.array_equal(ga["pt_xyz"], np.arange(3 * n, dtype=np.float64).reshape(n, 3)[rows.astype(np.int64)])
