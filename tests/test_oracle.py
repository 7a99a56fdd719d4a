"""
CPU tests (-m "not gpu"): the two oracles (numpy port in both summation orders, plain-C
restatement) against the golden fixtures frozen from the live reference, the pinning grid of
oracle/check_against_reference.py from its stored outputs, and that grid live where the reference is staged.

Tolerances: statistics, weight sums, Partitioner outputs and error strings are compared
bit-exactly.  Matrices from the numpy port are compared at relFro <= 1e-14 (f64) because
their GEMM bits depend on the OpenBLAS kernel of the host; the C oracle accumulates its
GEMMs in plain row order, so its matrices are held to relFro <= 1e-12 (f64) / 1e-5 (f32).
"""

import os
import subprocess
import sys

import numpy as np
import pytest

import check_against_reference
import golden_io
from cvmatrix_oracle import OracleCVMatrix, OraclePartitioner, pairwise_sum, rel_fro, sequential_colsum
import c_oracle

STATS = ("X_mean", "X_std", "Y_mean", "Y_std")
TOL = {"float64": 1e-12, "float32": 1e-5}
PIN_GRID = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pin_grid.npz")


def _unpack(method, res):
    if method == "training_statistics":
        return {}, res
    if method == "training_XTX_XTY":
        return {"XTX": res[0][0], "XTY": res[0][1]}, res[1]
    return {method.split("_")[1]: res[0]}, res[1]


def _check_numpy_oracle(name, order):
    spec, inp, fit, out = golden_io.case(name)
    m = OracleCVMatrix(*spec["flags"], ddof=spec["ddof"], dtype=np.dtype(spec["dtype"]).type, order=order)
    m.fit(inp["X"], inp["Y"], inp["w"])
    for attr in ("sum_X", "sum_Y", "sum_sq_X", "sum_sq_Y"):
        if attr in fit:
            assert np.array_equal(getattr(m, attr), fit[attr]), (name, attr)
    if "sum_w" in fit:
        assert m.sum_w == fit["sum_w"] and m.nnz_w == fit["num_nonzero_w"]
    assert rel_fro(m.XTX, fit["XTX"]) <= 1e-14
    for i, val in enumerate(inp["vals"]):
        for method in spec["methods"]:
            key = f"val{i}/{method}"
            try:
                res = getattr(m, method)(val)
            except ValueError as e:
                assert out.get(key + "/error") == str(e), (name, key, str(e))
                continue
            assert key + "/error" not in out, (name, key)
            mats, stats = _unpack(method, res)
            for s_name, s in zip(STATS, stats):
                if s is None:
                    assert f"{key}/{s_name}" not in out, (name, key, s_name)
                else:
                    g = out[f"{key}/{s_name}"]
                    assert s.dtype == g.dtype and np.array_equal(s, g, equal_nan=True), (name, key, s_name)
            for m_name, a in mats.items():
                g = out[f"{key}/{m_name}"]
                assert a.dtype == g.dtype and a.shape == g.shape
                if np.all(np.isfinite(g)):
                    assert rel_fro(a, g) <= (1e-14 if spec["dtype"] == "float64" else 1e-6), (name, key, m_name)


@pytest.mark.parametrize("order", ["numpy", "explicit"])
def test_numpy_oracle_matches_golden(order):
    for name in golden_io.case_names():
        _check_numpy_oracle(name, order)


def test_c_oracle_matches_golden():
    """The C restatement returns the full statistic set; compare each one the reference returned."""
    n_checked = 0
    for name in golden_io.case_names():
        spec, inp, fit, out = golden_io.case(name)
        m = c_oracle.COracle(*spec["flags"], ddof=spec["ddof"], dtype=spec["dtype"])
        m.fit(inp["X"], inp["Y"], inp["w"])
        tol = TOL[spec["dtype"]]
        for attr in ("sum_X", "sum_Y", "sum_sq_X", "sum_sq_Y"):
            if attr in fit:
                assert np.array_equal(getattr(m, attr)[:, : fit[attr].shape[1]], fit[attr]), (name, attr)
        if "sum_w" in fit:
            assert m.sum_w == fit["sum_w"] and m.nnz_w == fit["num_nonzero_w"]
        assert rel_fro(m.XTX, fit["XTX"]) <= tol
        for i, val in enumerate(inp["vals"]):
            for method in spec["methods"]:
                key = f"val{i}/{method}"
                if key + "/error" in out:
                    if "Response variables" in out[key + "/error"]:
                        continue
                    r = m.fold(val, True, spec["has_Y"])
                    want = 1 if "greater than zero" in out[key + "/error"] else 2
                    assert r["status"] == want, (name, key, r["status"])
                    continue
                r = m.fold(val, method != "training_XTY", spec["has_Y"] and method != "training_XTX")
                for s_name in STATS:
                    if f"{key}/{s_name}" in out:
                        assert np.array_equal(r[s_name], out[f"{key}/{s_name}"], equal_nan=True), (name, key, s_name)
                        n_checked += 1
                for m_name in ("XTX", "XTY"):
                    if f"{key}/{m_name}" in out and np.all(np.isfinite(out[f"{key}/{m_name}"])):
                        g = out[f"{key}/{m_name}"]
                        # a fold whose centred matrix is pure cancellation residue (one training row
                        # with non-zero weight) is held to the scale of the uncentred total instead
                        noise_floor = tol * np.linalg.norm(fit[m_name]) if not (spec["flags"][2] or spec["flags"][3]) else 0.0
                        err = np.linalg.norm(r[m_name].astype(np.float64) - g)
                        assert rel_fro(r[m_name], g) <= tol or err <= noise_floor, (name, key, m_name)
                        n_checked += 1
    assert n_checked > 1000


def test_partitioner_oracle_matches_golden():
    for pc in golden_io.manifest()["partitioner"]:
        folds = eval(pc["folds_repr"])  # noqa: S307 - fixture written by make_golden.py
        d = OraclePartitioner(folds).folds_dict
        assert [repr(k) for k in d] == pc["keys_repr"]
        for v, g in zip(d.values(), pc["indices"]):
            assert v.dtype == np.int64 and v.tolist() == g


def test_summation_orders_match_numpy():
    rng = np.random.default_rng(0)
    for dt in (np.float64, np.float32):
        for n in (0, 1, 7, 8, 9, 127, 128, 129, 1000, 4097, 100003):
            a = (rng.random(n) * rng.choice([1.0, 1e3], n)).astype(dt)
            ref = np.sum(a.reshape(-1, 1))
            assert pairwise_sum(a) == ref and c_oracle.pairwise_sum(a) == ref, (dt, n)
        for n, c in ((1, 2), (3, 5), (1000, 37), (200, 500), (50000, 3)):
            A = rng.random((n, c)).astype(dt)
            ref = np.sum(A, axis=0, keepdims=True)
            assert np.array_equal(sequential_colsum(A), ref)
            assert np.array_equal(c_oracle.colsum(A), ref)
        A = rng.random((777, 1)).astype(dt)
        assert np.array_equal(c_oracle.colsum(A), np.sum(A, axis=0, keepdims=True))


def test_oracle_matches_pinned_grid():
    """The pinning grid of oracle/check_against_reference.py, offline (tests/golden/pin_grid.npz): Partitioner outputs,
    statistics, weight sums and error messages bit for bit; matrices, whose bits depend on the host's BLAS, to
    relFro <= 1e-14 (float64) / 1e-6 (float32); both summation orders."""
    want, _ = check_against_reference.load_recorded(PIN_GRID)
    assert len(want) > 30_000
    for order in ("numpy", "explicit"):
        bad = check_against_reference.compare(check_against_reference.grid_outputs(*check_against_reference.oracle_classes(order)),
                                              want, matrix_tol=1e-14)
        assert not bad, (order, len(bad), bad[:10])


@pytest.mark.skipif(not os.path.isfile(os.path.join(check_against_reference.REF, "cvmatrix", "cvmatrix.py")),
                    reason="needs the unmodified reference: oracle/_ref staged by `make -C oracle ref`, or CVMATRIX_REFERENCE")
def test_oracle_pinned_to_live_reference():
    script = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "check_against_reference.py")
    r = subprocess.run([sys.executable, script], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_downdating_oracle_equals_naive_recomputation():
    """The reference's own test strategy (tests/test_cvmatrix.py:420-575): fast == naive for all 16 flag combinations,
    weighted (with zero weights) and unweighted, atol = 1e-8."""
    import itertools

    from cvmatrix_oracle import make_inputs
    from naive_oracle import naive_training_matrices

    X, Y, w, folds = make_inputs(700, 9, 3, 3, seed=31)
    w[::7] = 0
    for flags in itertools.product((False, True), repeat=4):
        for weights in (w, None):
            o = OracleCVMatrix(*flags)
            o.fit(X, Y, weights)
            for f in range(3):
                val = np.flatnonzero(folds == f)
                r = o.fold(val)
                n = naive_training_matrices(X, Y, weights, val, *flags)
                np.testing.assert_allclose(r.XTX, n["XTX"], atol=1e-8)
                np.testing.assert_allclose(r.XTY, n["XTY"], atol=1e-8)
                for name, got in (("X_mean", r.X_mean), ("X_std", r.X_std), ("Y_mean", r.Y_mean), ("Y_std", r.Y_std)):
                    if got is not None:
                        np.testing.assert_allclose(got, n[name], atol=1e-10)
