"""bench.py --dump-outputs: whole columns when they fit, else the same seeded sample of events every time, within
the byte budget."""
import os

import numpy as np

import bench


def _dump(d, n):
    rng = np.random.default_rng(7)
    per_event = {"round": rng.integers(0, 900, n, dtype=np.int32), "witness": rng.integers(0, 2, n, dtype=np.uint8),
                 "famous": rng.integers(-1, 2, n, dtype=np.int8)}
    tables = {"witness_table": rng.integers(-1, n, (40, 16), dtype=np.int32), "consensus": np.arange(30, dtype=np.int32)}
    bench.dump_outputs(str(d), n, per_event, tables)
    return per_event, tables, {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_whole_columns_when_they_fit(tmp_path):
    per_event, tables, got = _dump(tmp_path, 5000)
    assert set(got) == set(per_event) | set(tables)
    for k, v in {**per_event, **tables}.items():
        assert got[k].dtype == np.float32 and np.array_equal(got[k], v)


def test_seeded_sample_within_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    n = 200000
    per_event, tables, got = _dump(tmp_path / "a", n)
    idx = got["sample_index"].astype(np.int64)
    assert got["sample_index"].dtype == np.float64 and 0 < len(idx) < n
    assert np.all(np.diff(idx) > 0) and idx[-1] < n
    for k, v in per_event.items():
        assert np.array_equal(got[k], v[idx])
    for k, v in tables.items():
        assert np.array_equal(got[k], v)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 1 << 20
    again = _dump(tmp_path / "b", n)[2]
    assert all(np.array_equal(again[k], got[k]) for k in got)
