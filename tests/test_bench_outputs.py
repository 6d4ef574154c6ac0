"""CPU: the files `bench.py --dump-outputs DIR` writes, which two builds are compared by."""
import numpy as np

import bench


def test_outputs_are_float_npy_files(tmp_path):
    logits = np.random.default_rng(0).standard_normal((2, 1000)).astype(np.float32)
    ids = np.array([5, 2 ** 40 + 3], dtype=np.int64)
    bench.write_outputs(str(tmp_path), {"logits": logits, "next_ids": ids})
    assert sorted(p.name for p in tmp_path.iterdir()) == ["logits.npy", "next_ids.npy"]
    got_logits, got_ids = np.load(tmp_path / "logits.npy"), np.load(tmp_path / "next_ids.npy")
    assert got_logits.dtype == np.float32 and np.array_equal(got_logits, logits)
    assert got_ids.dtype == np.float64 and np.array_equal(got_ids.astype(np.int64), ids)


def test_large_output_is_the_same_sample_within_the_limit(tmp_path):
    limit = 1 << 20
    big = np.random.default_rng(1).standard_normal((64, 8192)).astype(np.float32)  # 2 MiB
    dumps = []
    for name in ("a", "b"):
        d = tmp_path / name
        bench.write_outputs(str(d), {"logits": big, "next_ids": np.arange(64)}, limit=limit)
        assert sum(p.stat().st_size for p in d.iterdir()) <= limit
        dumps.append((np.load(d / "logits.npy"), np.load(d / "logits_index.npy")))
    (vals, idx), (vals2, idx2) = dumps
    assert np.array_equal(idx, idx2) and np.array_equal(vals, vals2)
    assert np.all(np.diff(idx) > 0) and np.array_equal(vals, big.reshape(-1)[idx.astype(np.int64)])
    assert vals.size > 10_000
