"""bench.py --dump-outputs: what it writes, and the seeded row sample it falls back to above the size limit."""
import os

import numpy as np

import bench


def _arrays(E):
    rng = np.random.default_rng(3)
    return {"action": rng.standard_normal((E, 2)).astype(np.float32),
            "obs": rng.standard_normal((E, 15, 4)).astype(np.float32),
            "terminated": (rng.random(E) < 0.1).astype(np.uint8)}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_small_outputs_are_written_whole_as_float32(tmp_path):
    src = _arrays(100)
    bench.dump_outputs(str(tmp_path), src)
    got = _load(tmp_path)
    assert set(got) == set(src)
    for k, a in src.items():
        assert got[k].dtype == np.float32 and np.array_equal(got[k], a.astype(np.float32)), k


def test_large_outputs_keep_the_same_seeded_rows_under_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 64 << 10)
    src = _arrays(5000)
    runs = []
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), src)
        runs.append(_load(tmp_path / name))
        assert sum(os.path.getsize(tmp_path / name / f) for f in os.listdir(tmp_path / name)) <= 64 << 10
    a, b = runs
    assert set(a) == set(src) | {"env_index"} and a["env_index"].dtype == np.float64
    idx = a["env_index"].astype(np.int64)
    assert 0 < len(idx) < 5000 and np.all(np.diff(idx) > 0)
    for k in src:
        assert np.array_equal(a[k], src[k][idx].astype(np.float32)) and np.array_equal(a[k], b[k]), k
