"""bench.py --dump-outputs (no GPU needed): the sampled tracks are read through the tiled layout correctly, every array is
float32 or float64, and the files stay within 64 MB at the benchmark's shape."""
import os

import numpy as np
import torch

import bench
from em_model_manned_bayes_b200.model import TrackResult, tile


def test_dump_outputs_writes_the_sampled_tracks_of_the_result(tmp_path):
    rs = np.random.default_rng(5)
    n, T, n_dyn, n_tv, ni = 5003, bench.T, 3, 4, 7
    bins = rs.integers(1, 20, size=(n, n_dyn, T)).astype(np.int8)
    vals = rs.standard_normal((n, n_tv, T)).astype(np.float32)
    ib = rs.integers(1, 9, size=(ni, n)).astype(np.int8)
    iv = rs.standard_normal((ni, n))
    att = rs.integers(1, 65535, size=n).astype(np.uint16)
    res = TrackResult(n=n, T=T, dyn_vars=[1, 2, 3], tv_vars=[1, 2, 3, 4], bins_tiled=torch.from_numpy(tile(bins)),
                      values_tiled=torch.from_numpy(tile(vals)), init_bins=torch.from_numpy(ib), init_values=torch.from_numpy(iv),
                      attempts=torch.from_numpy(att.view(np.int16)))
    hi = torch.arange(ni * 64, dtype=torch.int64).reshape(ni, 64)
    ht = torch.arange(n_dyn * 64, dtype=torch.int64).reshape(n_dyn, 64)
    bench.dump_outputs(str(tmp_path), res, hi, ht)
    d = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)) <= 64 << 20
    idx = d["track_index"].astype(np.int64)
    assert len(idx) == bench.DUMP_TRACKS and np.all(np.diff(idx) > 0) and idx[-1] < n
    assert np.array_equal(d["bins"], bins[idx])
    assert np.array_equal(d["values"], vals[idx])
    assert np.array_equal(d["init_bins"], ib[:, idx])
    assert np.array_equal(d["init_values"], iv[:, idx])
    assert np.array_equal(d["attempts"], att[idx])
    assert np.array_equal(d["hist_initial"], hi.numpy()) and np.array_equal(d["hist_transition"], ht.numpy())
    bench.dump_outputs(str(tmp_path / "again"), res, hi, ht)
    assert np.array_equal(np.load(os.path.join(tmp_path, "again", "track_index.npy")), d["track_index"])
