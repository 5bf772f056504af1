"""``bench.py --dump-outputs``: file names, dtypes, and the seeded sample kept when the outputs
exceed the size cap (no GPU; the arrays stand in for v and status)."""

import os

import numpy as np

import bench


def _dump(tmp_path, B, limit, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT", limit)
    v = np.arange(B * 6, dtype=np.float32).reshape(B, 6)
    status = (np.arange(B) % 3).astype(np.int32)
    bench.dump_outputs(str(tmp_path), {"v": v, "status": status})
    names = sorted(os.listdir(tmp_path))
    return names, {n[:-4]: np.load(os.path.join(tmp_path, n)) for n in names}


def test_small_outputs_are_written_whole(tmp_path, monkeypatch):
    names, out = _dump(tmp_path, 1000, 1 << 20, monkeypatch)
    assert names == ["status.npy", "v.npy"]
    assert out["v"].dtype == np.float32 and out["status"].dtype == np.float32
    np.testing.assert_array_equal(out["v"], np.arange(6000, dtype=np.float32).reshape(1000, 6))
    np.testing.assert_array_equal(out["status"], np.arange(1000) % 3)


def test_large_outputs_keep_one_seeded_sample_under_the_cap(tmp_path, monkeypatch):
    limit, B = 200_000, 100_000
    names, out = _dump(tmp_path / "a", B, limit, monkeypatch)
    assert names == ["instance.npy", "status.npy", "v.npy"]
    assert sum(os.path.getsize(os.path.join(tmp_path / "a", n)) for n in names) <= limit
    rows = out["instance"]
    assert rows.dtype == np.float64 and (np.diff(rows) > 0).all() and rows[-1] < B
    assert len(rows) > 0.9 * limit / (6 * 4 + 4 + 8)  # the cap is nearly used
    idx = rows.astype(np.int64)
    np.testing.assert_array_equal(out["v"][:, 0], 6 * idx)  # every array keeps the same instances
    np.testing.assert_array_equal(out["status"], idx % 3)
    _, again = _dump(tmp_path / "b", B, limit, monkeypatch)
    np.testing.assert_array_equal(again["instance"], rows)  # fixed seed: the same sample every run
