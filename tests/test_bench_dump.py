"""bench.py --dump-outputs: the result of the last timed step as float64 arrays, rows in key order (no GPU needed)."""
import numpy as np

import bench

KEYS = ["labels.a", "labels.b"]
AGGS = ["sum(value)", "count(value)"]


def load(d):
    return {p.name: np.load(p) for p in sorted(d.iterdir())}


def test_dump_outputs_writes_one_float64_array_per_column_in_key_order(tmp_path):
    rows = {(("labels.a", "y"), ("labels.b", "z")): (None, 0),
            (("labels.a", "x"), ("labels.b", "z")): (5, 1),
            (("labels.a", "y"), ("labels.b", None)): (7, 2)}
    bench.dump_outputs(str(tmp_path), rows, KEYS, AGGS)
    out = load(tmp_path)
    assert sorted(out) == ["count_value.npy", "labels.a.npy", "labels.b.npy", "sum_value.npy"]
    assert all(a.dtype == np.float64 and a.shape == (3,) for a in out.values())
    # key order, NULL last: (x, z), (y, z), (y, NULL)
    np.testing.assert_array_equal(out["sum_value.npy"], [5, np.nan, 7])
    np.testing.assert_array_equal(out["count_value.npy"], [1, 0, 2])
    a, b = out["labels.a.npy"], out["labels.b.npy"]
    assert a[1] == a[2] != a[0] and b[0] == b[1] and np.isnan(b[2])
    assert all(v == int(v) and 0 <= v < 2 ** 48 for v in (a[0], a[1], b[0]))


def test_dump_outputs_samples_a_large_result_the_same_way_every_time(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 8 * 4 * 10)  # ten rows of four columns
    rows = {(("labels.a", f"v{i:03d}"), ("labels.b", f"w{i % 7}")): (i, 1) for i in range(100)}
    bench.dump_outputs(str(tmp_path / "1"), dict(reversed(list(rows.items()))), KEYS, AGGS)
    bench.dump_outputs(str(tmp_path / "2"), rows, KEYS, AGGS)
    first, second = load(tmp_path / "1"), load(tmp_path / "2")
    for name, arr in first.items():
        np.testing.assert_array_equal(arr, second[name])
    s = first["sum_value.npy"]
    assert s.shape == (10,) and (np.diff(s) > 0).all()  # a subset of the rows, still in key order
