"""bench.py --dump-outputs (no GPU): the last timed step's results land as float .npy files that hold the same values."""
import numpy as np

import bench


def test_dump_outputs_writes_float_arrays_with_the_same_values(tmp_path):
    sc = np.array([[-1.5, -2.25], [-0.5, -3.0]], np.float32)
    ids = np.array([[7, (1 << 40) + 3], [2, -1]], np.int64)
    cnt = np.array([2, 1], np.int32)
    out = tmp_path / "dump"
    bench.dump_outputs(str(out), "c5", sc, ids, cnt)
    assert sorted(p.name for p in out.iterdir()) == ["c5_counts.npy", "c5_ids.npy", "c5_scores.npy"]
    got_sc, got_ids, got_cnt = (np.load(out / f"c5_{p}.npy") for p in ("scores", "ids", "counts"))
    assert got_sc.dtype == np.float32 and got_ids.dtype == np.float64 and got_cnt.dtype == np.float64
    np.testing.assert_array_equal(got_sc, sc)
    np.testing.assert_array_equal(got_ids.astype(np.int64), ids)
    np.testing.assert_array_equal(got_cnt, cnt)


def test_no_directory_writes_nothing(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    bench.dump_outputs(None, "c5", np.zeros((1, 1), np.float32), np.zeros((1, 1), np.int64), np.zeros(1, np.int32))
    assert list(tmp_path.iterdir()) == []
