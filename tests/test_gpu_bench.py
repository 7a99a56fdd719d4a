"""GPU test (-m gpu) of the native bench.py arm on the tiny self-test shape: one JSON line with the contract's keys,
kernels actually launched, e2e measured through the public API with host buffers."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_native_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "tiny", "--steps", "3", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in d, key
    assert d["metric"] == "fold matrices/sec" and d["unit"] == "fold-matrices/s" and d["n_gpus"] == 1 and d["dtype"] == "f64"
    assert d["value"] > 0 and d["gpu_launches"] > 0 and d["steps"] == 3 and d["warmup"] == 3
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    roof = d["roofline"]
    assert roof["bound"] in ("hbm", "tensor") and roof["peak"] > 0 and roof["achieved"] > 0 and roof["kernel"].startswith("k_gram")
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] > 0 and d["cpu_baseline"]["cores"] >= 1
    par = d["parity"]
    assert par["stats_bit_exact"] is True and par["xtx"] <= 1e-12 and par["xty"] <= 1e-12 and par["joint"] <= 1e-12 and par["folds_checked"] == 4
    assert d["parity_e2e_path"]["stats_bit_exact"] is True and d["parity_e2e_path"]["joint"] <= 1e-12



@pytest.mark.parametrize("config, N, K, M, P", [("tiny", 4_000, 24, 3, 4), ("cfg4", 20_000, 500, 10, 20_000)])
def test_dump_outputs_of_the_timed_step(tmp_path, config, N, K, M, P):
    """--dump-outputs writes what training_batch returns for the folds of the last timed step, float64, under 64 MB, and
    they equal the numpy oracle on the same seeded inputs.  tiny: every fold.  cfg4 (leave-one-out, 20 000 folds in output
    windows of 4096): a seeded sample of the last window, folds 16384..19999."""
    from cvmatrix_oracle import OracleCVMatrix, make_inputs, rel_fro

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", config, "--steps", "2", "--warmup", "3",
                        "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    names = {"XTX", "XTY", "X_mean", "X_std", "Y_mean", "Y_std", "sum_w_train", "nnz_train", "status", "folds", "rows"}
    assert {p.name for p in tmp_path.iterdir()} == {n + ".npy" for n in names}
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64_000_000
    d = {n: np.load(tmp_path / (n + ".npy")) for n in names}
    assert all(a.dtype == np.float64 for a in d.values())
    folds = d["folds"].astype(np.int64)
    assert np.array_equal(d["rows"], np.arange(K))
    if P <= 4096:
        assert np.array_equal(folds, np.arange(P))
    else:
        assert folds.size >= 16 and np.all(np.diff(folds) > 0) and folds[0] >= 16_384 and folds[-1] < P
    assert d["XTX"].shape == (folds.size, K, K) and d["XTY"].shape == (folds.size, K, M) and d["X_mean"].shape == (folds.size, 1, K)
    X, Y, w, labels = make_inputs(N, K, M, P)   # the inputs bench.py generates
    orc = OracleCVMatrix(copy=False)
    orc.fit(X, Y, w)
    for i, f in enumerate(folds):
        o = orc.fold(np.flatnonzero(labels == f))
        assert rel_fro(d["XTX"][i], o.XTX) <= 1e-12 and rel_fro(d["XTY"][i], o.XTY) <= 1e-12, f
        for s in ("X_mean", "X_std", "Y_mean", "Y_std"):
            assert np.array_equal(d[s][i], getattr(o, s)), (f, s)
        assert d["sum_w_train"][i] == o.sum_w_train and d["nnz_train"][i] == o.nnz_train, f
    assert not d["status"].any()
