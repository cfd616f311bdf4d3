"""bench.py's host logic that needs no GPU: what --dump-outputs writes, and the --steps argument."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_writes_float_arrays_whole_for_small_clouds(tmp_path):
    P = 40
    rng = np.random.default_rng(1)
    img, radii, grad = rng.normal(size=(2, 3, 4, 5)).astype(np.float32), rng.integers(0, 9, (P, 2)).astype(np.int32), rng.normal(size=(P, 3))
    bench.dump_outputs(str(tmp_path), P, {"color": img}, {"radii": radii, "dL_dmeans3D": grad})
    out = _load(tmp_path)
    assert sorted(out) == ["color", "dL_dmeans3D", "radii"]
    assert out["color"].dtype == np.float32 and np.array_equal(out["color"], img)
    assert out["radii"].dtype == np.float32 and np.array_equal(out["radii"], radii)
    assert out["dL_dmeans3D"].dtype == np.float64 and np.array_equal(out["dL_dmeans3D"], grad)


def test_dump_samples_the_same_gaussians_every_time(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 16)
    P = 100
    grad = np.arange(P * 3, dtype=np.float32).reshape(P, 3)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), P, {}, {"dL_dscales": grad})
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    idx = a["gaussian_index"]
    assert idx.dtype == np.float64 and idx.shape == (16,) and np.all(np.diff(idx) > 0) and idx[-1] < P
    assert np.array_equal(a["dL_dscales"], grad[idx.astype(np.int64)])
    assert all(np.array_equal(a[k], b[k]) for k in a)


def test_dump_refuses_more_than_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 1000)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "x"), 10, {"color": np.zeros(251, np.float32)}, {})
    assert not (tmp_path / "x").exists()


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, bench.__file__, "--steps", "0"], capture_output=True, text=True)
    assert r.returncode == 2 and "--steps" in r.stderr
