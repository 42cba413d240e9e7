"""bench.py --dump-outputs: what it writes, within its byte budget, identically from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(d, names):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in names}


def test_write_outputs_whole_and_sampled(tmp_path):
    rng = np.random.default_rng(0)
    per_point = {"mean": rng.standard_normal(1000), "var": rng.uniform(size=1000)}
    other = {"pce_mean": np.array([0.25])}
    full = str(tmp_path / "full")
    bench.write_outputs(full, per_point, other)
    got = _load(full, ["mean", "var", "pce_mean"])
    assert sorted(os.listdir(full)) == ["mean.npy", "pce_mean.npy", "var.npy"]
    for k, v in {**per_point, **other}.items():
        assert got[k].dtype == np.float64 and np.array_equal(got[k], v)

    cuts = []
    for i in range(2):                             # the same sample every time
        d = str(tmp_path / ("cut%d" % i))
        bench.write_outputs(d, per_point, other, max_bytes=8000, suffix="_rank1")
        assert sorted(os.listdir(d)) == ["index_rank1.npy", "mean_rank1.npy", "pce_mean_rank1.npy", "var_rank1.npy"]
        assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= 8000
        cuts.append({k: np.load(os.path.join(d, k + "_rank1.npy")) for k in ("index", "mean", "var", "pce_mean")})
    a, b = cuts
    idx = a["index"].astype(np.int64)
    assert len(idx) > 200 and np.all(np.diff(idx) > 0) and np.array_equal(idx, a["index"])
    assert np.array_equal(a["mean"], per_point["mean"][idx]) and np.array_equal(a["var"], per_point["var"][idx])
    assert a["pce_mean"][0] == 0.25
    for k in a:
        assert np.array_equal(a[k], b[k])


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_steps_results_and_repeat(gpu, tmp_path):
    """Two runs with the same arguments dump the same bits; the dumped PCE mean is the one the JSON line
    reports and the quadrature-weighted sum of the dumped means."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--points", "4096",
           "--samples", "16", "--nh", "256", "--nl", "1024", "--no-lml", "--no-cpu", "--no-extras"]
    runs = []
    for i in range(2):
        d = str(tmp_path / str(i))
        r = subprocess.run(cmd + ["--dump-outputs", d], capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
        assert r.returncode == 0, r.stderr[-4000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and line["warmup"] == 1
        assert sorted(os.listdir(d)) == ["mean.npy", "pce_mean.npy", "var.npy"]
        runs.append((line, _load(d, ["mean", "var", "pce_mean"])))
    (line, a), (_, b) = runs
    for k in a:
        assert a[k].dtype == np.float64 and np.array_equal(a[k], b[k]), k
    assert a["mean"].shape == a["var"].shape == (4096,)
    assert np.isfinite(a["mean"]).all() and (a["var"] > 0).all()
    assert a["pce_mean"].shape == (1,) and a["pce_mean"][0] == line["pce_mean"]
    _, w = bench.gauss_legendre_grid(8, 4)
    assert np.isclose(a["pce_mean"][0], np.sum(w * a["mean"]), rtol=1e-12)
