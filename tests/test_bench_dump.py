"""CPU: bench.py --dump-outputs writes what it was given whole while it fits, stays within its size budget when it does not,
and stores the same elements on every run."""
import os

import numpy as np

import bench


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_whole_when_it_fits(tmp_path):
    rng = np.random.default_rng(1)
    arrays = {"total": np.float32(2.5), "terms": rng.standard_normal((4, 6)),
              "grad_W1": rng.standard_normal((4, 6, 8, 19)).astype(np.float16)}
    bench.dump_outputs(str(tmp_path), arrays)
    got = _load(tmp_path)
    assert set(got) == set(arrays)
    assert got["terms"].dtype == np.float64 and np.array_equal(got["terms"], arrays["terms"])
    assert got["grad_W1"].dtype == np.float32 and np.array_equal(got["grad_W1"], arrays["grad_W1"].astype(np.float32))
    assert got["total"].shape == () and got["total"] == np.float32(2.5)


def test_dump_outputs_budget_and_repeatability(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    rng = np.random.default_rng(2)
    arrays = {"terms": rng.standard_normal((8, 6)), "grad_W2": rng.standard_normal((8, 6, 64, 256)).astype(np.float32),
              "grad_Wa": rng.standard_normal(1 << 18)}
    runs = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= 1 << 20
        runs.append(_load(tmp_path / d))
    a, b = runs
    assert np.array_equal(a["terms"], arrays["terms"])
    flat = arrays["grad_W2"].reshape(-1)
    assert a["grad_W2"].ndim == 1 and 0 < a["grad_W2"].size < flat.size and np.isin(a["grad_W2"], flat).all()
    assert a["grad_Wa"].dtype == np.float64 and np.isin(a["grad_Wa"], arrays["grad_Wa"]).all()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
