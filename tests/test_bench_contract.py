"""bench.py contract: the reference arm (CPU only) prints one JSON line with the agreed keys; the native arm refuses
to run without a GPU instead of falling back."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "tiny", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "fold matrices/sec" and d["unit"] == "fold-matrices/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["steps_requested"] == 2 and d["cpu_baseline"]["blas_threads"] >= 1
    assert set(d["config"]) >= {"workload", "N", "K", "M", "folds", "parallelism", "step"}
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "tiny", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_native_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "tiny", "--steps", "1"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)



def test_argument_checks():
    """Refused before any work: a step count below one, and --dump-outputs outside the native single-process path."""
    for extra, msg in ((("--steps", "0"), "--steps must be at least 1"),
                       (("--impl", "reference", "--dump-outputs", "unused"), "--dump-outputs writes the native path's results")):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "tiny", *extra], capture_output=True,
                           text=True, timeout=120)
        assert r.returncode == 2 and msg in r.stderr, (extra, r.stderr[-2000:])


@pytest.fixture
def bench(monkeypatch):
    """bench.py as a module; the thread-count variables it sets on import are restored afterwards."""
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        monkeypatch.setenv(v, os.environ.get(v, ""))
    monkeypatch.syspath_prepend(ROOT)
    import bench

    return bench


@pytest.mark.parametrize("n, K, M, first", [(3, 24, 3, 0), (40, 500, 10, 16_384), (2, 3_000, 10, 7)])
def test_dump_outputs_sampling(bench, tmp_path, n, K, M, first):
    """dump_outputs on CPU tensors: every fold and row when they fit, else a seeded sample of the folds (and of the XTX / XTY
    rows when one fold alone is too large), always under 64 MB and equal to the entries it names."""
    import torch

    g = torch.Generator().manual_seed(1)
    outs = dict(XTX=torch.rand((n, K, K), generator=g, dtype=torch.float64), XTY=torch.rand((n, K, M), generator=g, dtype=torch.float64),
                stats=torch.rand((n, 2, K + M), generator=g, dtype=torch.float64), scal=torch.rand((n, 2), generator=g, dtype=torch.float64),
                status=torch.arange(n, dtype=torch.int32))
    bench.dump_outputs(str(tmp_path), outs, first, n, K)
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64_000_000
    d = {p.name[:-4]: np.load(p) for p in tmp_path.iterdir()}
    assert all(a.dtype == np.float64 for a in d.values())
    pos, rows = d["folds"].astype(np.int64) - first, d["rows"].astype(np.int64)
    per_fold = 8 * (K * K + K * M + 2 * (K + M) + 3)
    assert pos.size == (n if n * per_fold <= bench.DUMP_LIMIT_BYTES else max(1, bench.DUMP_LIMIT_BYTES // per_fold))
    assert rows.size == (K if per_fold <= bench.DUMP_LIMIT_BYTES else bench.DUMP_LIMIT_BYTES // (16 * (K + M)))
    assert np.all(np.diff(pos) > 0) and 0 <= pos[0] and pos[-1] < n and np.all(np.diff(rows) > 0) and rows[-1] < K
    st = outs["stats"].numpy()[pos]
    assert np.array_equal(d["XTX"], outs["XTX"].numpy()[pos][:, rows]) and np.array_equal(d["XTY"], outs["XTY"].numpy()[pos][:, rows])
    assert np.array_equal(d["X_std"], st[:, 1:2, :K]) and np.array_equal(d["Y_mean"], st[:, 0:1, K:])
    assert np.array_equal(d["nnz_train"], outs["scal"].numpy()[pos, 1]) and np.array_equal(d["status"], pos)
    again = tmp_path / "again"
    bench.dump_outputs(str(again), outs, first, n, K)
    assert all(np.array_equal(np.load(again / (k + ".npy")), v) for k, v in d.items())
