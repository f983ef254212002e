"""bench.py --dump-outputs without a GPU: dtypes, whole arrays at the default pool size, and the size cap with one fixed
sample of rows shared by every array."""
import os

import numpy as np

import bench


def test_dump_outputs_writes_whole_arrays(tmp_path):
    rng = np.random.default_rng(0)
    a = dict(N=rng.integers(0, 600, (bench.TREES_PER_GPU, 7)), W=rng.normal(size=(bench.TREES_PER_GPU, 7)),
             P=rng.random((bench.TREES_PER_GPU, 7), dtype=np.float32))
    bench.dump_outputs(str(tmp_path), a, 0, 1)
    assert sorted(os.listdir(tmp_path)) == ["N.npy", "P.npy", "W.npy"]
    for k, v in a.items():
        x = np.load(tmp_path / (k + ".npy"))
        assert x.dtype == (np.float32 if k == "P" else np.float64) and (x == v).all()


def test_dump_outputs_caps_the_size_with_a_fixed_row_sample(tmp_path):
    S, world = 300000, 2
    rows = np.repeat(np.arange(S)[:, None], 7, axis=1)     # every value names its row
    a = dict(N=rows, W=rows.astype(np.float64), P=rows.astype(np.float32))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), a, 1, world)
    assert sorted(os.listdir(tmp_path / "a")) == ["N_rank1.npy", "P_rank1.npy", "W_rank1.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_BYTES // world + 3 * 128
    kept = np.load(tmp_path / "a" / "N_rank1.npy")[:, 0]
    assert 0 < len(kept) < S and (np.diff(kept) > 0).all()
    for f in os.listdir(tmp_path / "a"):
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert (x == y).all() and (x[:, 0] == kept).all()
