"""
GPU tests (-m gpu) of the out-of-fold predictions of cross-validated PLS and ridge (return_predictions=True;
cvmx_pls_cv_predict / cvmx_ridge_cv_predict): against the numpy oracles on the engine's own training matrices and
statistics, against the same call's B and PRESS, bit-identical other outputs with and without predictions, host and
device outputs over windows, passes and staged PRESS launches, the special rows (refused folds, failed pairs, early
stops, empty folds, repeated and negative indices), scikit-learn's cross_val_predict, and streams.
"""

import os
import re

import numpy as np
import pytest

import pls_oracle as po
import ridge_oracle as ro

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = np.finfo(np.float64).eps
C_RIDGE = 50.0
PRESS_ROWS = 32


def _stage_bytes():
    """CV_PRED_STAGE_BYTES of csrc/kernels_pls.cuh: the device bytes that stage one PRESS launch's host predictions."""
    src = open(os.path.join(ROOT, "cvmatrix_b200", "csrc", "kernels_pls.cuh")).read()
    a, b = re.search(r"CV_PRED_STAGE_BYTES = \(int64_t\)(\d+) << (\d+);", src).groups()
    return int(a) << int(b)


def _inputs(N, K, M, seed, weighted=True, dtype=np.float64):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, K)) + rng.standard_normal(K)
    Cm = rng.standard_normal((K, M)) * (0.8 ** np.minimum(np.arange(M), 20))
    Y = X @ Cm / np.sqrt(K) + 0.5 * rng.standard_normal((N, M)) + 1.0
    w = None
    if weighted:
        w = rng.random(N) + 0.1
        w[::7] = 0.0
    return X.astype(dtype), Y.astype(dtype), (None if w is None else w.astype(dtype))


def _model(X, Y, w, flags=15, dtype=np.float64, folds=None, sets=None):
    from cvmatrix_b200 import CVMatrix, Partitioner

    m = CVMatrix(center_X=bool(flags & 1), center_Y=bool(flags & 2), scale_X=bool(flags & 4), scale_Y=bool(flags & 8),
                 dtype=dtype)
    m.fit(X, Y, w)
    m.set_folds(sets if sets is not None else Partitioner(folds))
    return m


def _np(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else x


def _rel(a, b):
    b = np.asarray(b)
    nb = float(np.sqrt((b.astype(np.longdouble) ** 2).sum()))
    d = float(np.sqrt(((np.asarray(a).astype(np.longdouble) - b) ** 2).sum()))
    return d / (nb if nb > 0 else 1.0)


def _span(m, f, f0=0):
    """Rows of the predictions of a call over [f0, ..) that belong to fold f."""
    o = m._offsets
    return slice(int(o[f] - o[f0]), int(o[f + 1] - o[f0]))


def _stats(m, tb, i):
    g = lambda k: None if tb[k] is None else tb[k][i].astype(np.float64)  # noqa: E731
    return po.fold_stats(m._flags, g("X_mean"), g("X_std"), g("Y_mean"), g("Y_std"))


def _check_rows(m, r, f0, f1):
    idx = m._fold_indices[m._offsets[f0]:m._offsets[f1]]
    rows = _np(r["rows"])
    assert rows.dtype == np.int64 and np.array_equal(rows, np.where(idx < 0, idx + m.N, idx))


def _same(a, b, keys):
    for k in keys:
        x, y = _np(a[k]), _np(b[k])
        assert x.dtype == y.dtype and x.shape == y.shape, k
        assert np.array_equal(x, y, equal_nan=np.issubdtype(x.dtype, np.floating)), k


PLS_KEYS = ("press", "sum_w_val", "n_fitted", "status")
RIDGE_KEYS = ("press", "sum_w_val", "info", "status")


def _check_self_consistent(m, r, X, Y, w, f0=0, f1=None, dtype=np.float64):
    """Predictions against ((x - mu) / sigma) B sigma_Y + mu_Y from the same call's B, and every fold's press against
    sum w (y - pred)^2 recomputed from the returned predictions."""
    f1 = m._n_folds if f1 is None else f1
    tb = m.training_batch(f0, f1, check=False)
    pred = _np(r["predictions"]).astype(np.float64)
    for i in range(f1 - f0):
        f = f0 + i
        val = m._fold_indices[m._offsets[f]:m._offsets[f + 1]]
        if val.size == 0 or np.isnan(_np(r["press"])[i]).all():
            continue
        P = pred[_span(m, f, f0)].transpose(1, 0, 2)                 # [A or L, n, M]
        if dtype == np.float64 and r.get("B") is not None:
            ref = po.predict(X[val], _np(r["B"])[i], *_stats(m, tb, i))
            ok = ~np.isnan(ref).any(axis=(1, 2))
            assert _rel(P[ok], ref[ok]) <= 1e-13, (f, _rel(P[ok], ref[ok]))
        wv = np.ones(val.size) if w is None else w[val].astype(np.float64)
        res = Y[val].astype(np.float64)[None] - P
        pr = np.einsum("n,anm->am", wv, res * res)
        got = _np(r["press"])[i].astype(np.float64)
        ok = ~np.isnan(got)
        if dtype == np.float64:
            assert _rel(got[ok], pr[ok]) <= 1e-12, (f, _rel(got[ok], pr[ok]))
        else:
            # the kernel's residuals use the float64 predictions; the returned ones are rounded once to float32
            d = 2.0 ** -24 * np.abs(P) * 1.01
            bound = np.einsum("n,anm->am", wv, (2 * np.abs(res) + d) * d) + 2.0 ** -23 * np.abs(pr) + 1e-30
            assert (np.abs(got - pr)[ok] <= bound[ok]).all(), f


# ---- 1. PLS against the oracle, and self-consistency ---------------------------------------------------------------
@pytest.mark.parametrize("K", [64, 300])
@pytest.mark.parametrize("M", [1, 3, 40])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["float64", "float32"])
def test_pls_predictions_against_oracle(K, M, dtype):
    X, Y, w = _inputs(900, K, M, seed=K + M, dtype=dtype)
    P, A = 5, 15
    m = _model(X, Y, w, dtype=dtype, folds=np.arange(900) % P)
    r = m.pls_cross_validate(A, return_coefs=True, return_predictions=True)
    pred = r["predictions"]
    assert pred.shape == (900, A, M) and pred.dtype == dtype
    _check_rows(m, r, 0, P)
    tb = m.training_batch()
    tol = 1e-10 if dtype == np.float64 else 2e-5
    X64 = X.astype(np.float64)
    for f in range(P):
        val = m._fold_indices[m._offsets[f]:m._offsets[f + 1]]
        B, nf = po.ikpls(tb["XTX"][f], tb["XTY"][f], A)
        assert r["n_fitted"][f] == nf
        ref = po.predict(X64[val], B, *_stats(m, tb, f))
        got = pred[_span(m, f)].transpose(1, 0, 2)
        for a in range(A):
            assert _rel(got[a], ref[a]) <= tol, (f, a, _rel(got[a], ref[a]))
    _check_self_consistent(m, r, X, Y, w, dtype=dtype)


@pytest.mark.parametrize("flags", range(16))
def test_pls_predictions_all_flag_combinations(flags):
    X, Y, w = _inputs(120, 10, 2, seed=100 + flags)
    m = _model(X, Y, w, flags=flags, folds=np.arange(120) % 4)
    r = m.pls_cross_validate(5, return_coefs=True, return_predictions=True)
    tb = m.training_batch()
    for f in range(4):
        val = m._fold_indices[m._offsets[f]:m._offsets[f + 1]]
        B, _ = po.ikpls(tb["XTX"][f], tb["XTY"][f], 5)
        ref = po.predict(X[val], B, *_stats(m, tb, f))
        assert _rel(r["predictions"][_span(m, f)].transpose(1, 0, 2), ref) <= 1e-10, f
    _check_self_consistent(m, r, X, Y, w)


# ---- 1. ridge against the extended-precision oracle ----------------------------------------------------------------
def _scale(m):
    XTX = m.training_batch(0, 1)["XTX"][0].astype(np.float64)
    return np.trace(XTX) / XTX.shape[0]


def _compare_ridge_pred(m, r, X, alphas, f0=0, f1=None, cols=None, extra=0.0):
    """Predictions of folds [f0, f1) to C_RIDGE kappa eps64 of ridge_extended + predict in np.longdouble, per penalty;
    failed pairs NaN.  `cols`: the penalties of r that `alphas` are (default: all)."""
    f1 = m._n_folds if f1 is None else f1
    tb = m.training_batch(f0, f1, check=False)
    pred = _np(r["predictions"])
    cl = np.arange(len(alphas)) if cols is None else np.asarray(cols)
    for i in range(f1 - f0):
        f = f0 + i
        val = m._fold_indices[m._offsets[f]:m._offsets[f + 1]]
        if val.size == 0:
            continue
        XTX = tb["XTX"][i].astype(np.float64)
        B, info = ro.ridge_extended(XTX, tb["XTY"][i], alphas)
        ev = np.linalg.eigvalsh(XTX)
        ref = ro.predict(X[val], np.where(np.isnan(B), 0, B), *_stats(m, tb, i), dtype=np.longdouble)
        got = pred[_span(m, f, f0)]
        for l, c in enumerate(cl):
            g = got[:, c]
            if info[l]:
                assert np.isnan(g).all(), (f, l)
                continue
            kappa = (ev[-1] + alphas[l]) / (ev[0] + alphas[l])
            bound = C_RIDGE * kappa * EPS
            assert bound <= 1e-8, (f, l, kappa)
            e = _rel(g, ref[l])
            assert e <= bound + extra, (f, l, e, bound)


@pytest.mark.parametrize("K,M,dtype", [(20, 3, np.float64), (65, 1, np.float64), (130, 7, np.float64), (65, 1, np.float32),
                                       (130, 7, np.float32)])
def test_ridge_predictions_against_oracle(K, M, dtype):
    N, P = 3 * K + 90, 4
    X, Y, w = _inputs(N, K, M, seed=700 + K + M, dtype=dtype)
    m = _model(X, Y, w, dtype=dtype, folds=np.arange(N) % P)
    a = np.logspace(-2, 2, 5) * _scale(m)
    r = m.ridge_cross_validate(a, return_coefs=True, return_predictions=True)
    assert r["predictions"].shape == (N, 5, M) and r["predictions"].dtype == dtype
    _check_rows(m, r, 0, P)
    _compare_ridge_pred(m, r, X.astype(np.float64), a, extra=0.0 if dtype == np.float64 else 2e-6)
    _check_self_consistent(m, r, X, Y, w, dtype=dtype)


# ---- 3. nothing else moves -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("out", ["numpy", "torch"])
def test_other_outputs_bit_identical(out):
    X, Y, w = _inputs(300, 20, 3, seed=31)
    X[:, 13] = 0.0   # lam = 0 fails on every fold: info != 0 pairs are part of the comparison
    m = _model(X, Y, w, flags=3, folds=np.arange(300) % 5)
    a = [0.0, 0.5, 4.0]
    with pytest.warns(UserWarning):
        r0 = m.ridge_cross_validate(a, return_coefs=True, out=out)
    with pytest.warns(UserWarning):
        r1 = m.ridge_cross_validate(a, return_coefs=True, out=out, return_predictions=True)
    assert "predictions" not in r0 and "rows" not in r0
    _same(r0, r1, RIDGE_KEYS + ("B",))
    X2, Y2, w2 = _inputs(300, 20, 3, seed=32)
    m2 = _model(X2, Y2, w2, folds=np.arange(300) % 5)
    p0 = m2.pls_cross_validate(8, return_coefs=True, out=out)
    p1 = m2.pls_cross_validate(8, return_coefs=True, out=out, return_predictions=True)
    _same(p0, p1, PLS_KEYS + ("B",))
    if out == "torch":
        assert p1["predictions"].is_cuda and p1["rows"].is_cuda and r1["predictions"].is_cuda


# ---- 4. windows, passes and staged launches ------------------------------------------------------------------------
def test_pls_predictions_over_windows():
    # leave-one-out, K = 256: 2500 folds take two ~1 GiB windows (the first ends near fold 1945)
    X, Y, w = _inputs(2500, 256, 2, seed=77)
    m = _model(X, Y, w, folds=np.arange(2500))
    rh = m.pls_cross_validate(4, fold_begin=3, return_predictions=True)
    rd = m.pls_cross_validate(4, fold_begin=3, return_predictions=True, out="torch")
    _same(rh, rd, PLS_KEYS + ("predictions", "rows"))
    assert rh["predictions"].shape == (2497, 4, 2)
    for f0, f1 in ((1940, 1941), (1950, 1951), (1930, 1960)):
        rf = m.pls_cross_validate(4, fold_begin=f0, fold_end=f1, return_predictions=True)
        assert np.array_equal(rf["predictions"], rh["predictions"][f0 - 3:f1 - 3]), (f0, f1)
    _check_self_consistent(m, m.pls_cross_validate(4, fold_begin=1930, fold_end=1960, return_coefs=True,
                                                   return_predictions=True), X, Y, w, 1930, 1960)


def test_ridge_predictions_over_windows():
    # leave-one-out over 600 rows, folds 5 .. 599: four windows of ~189 folds for host and for device outputs
    K, M, L, N, f0 = 200, 8, 16, 600, 5
    X, Y, w = _inputs(N, K, M, seed=600)
    m = _model(X, Y, w, folds=np.arange(N))
    a = np.logspace(-2, 2, L) * _scale(m)
    rh = m.ridge_cross_validate(a, fold_begin=f0, return_predictions=True)
    rd = m.ridge_cross_validate(a, fold_begin=f0, return_predictions=True, out="torch")
    _same(rh, rd, RIDGE_KEYS + ("predictions", "rows"))
    for g0, g1 in ((180, 181), (190, 191), (175, 200)):
        rs = m.ridge_cross_validate(a, fold_begin=g0, fold_end=g1, return_predictions=True)
        assert np.array_equal(rs["predictions"], rh["predictions"][g0 - f0:g1 - f0]), (g0, g1)
    _compare_ridge_pred(m, m.ridge_cross_validate(a, fold_begin=180, fold_end=192, return_predictions=True), X, a, 180, 192)


def test_ridge_predictions_over_passes():
    # K = 400, L = 1024: every fold is its own window and its penalties go in passes, so every PRESS launch writes a
    # strided column slice of the caller's rows
    K, M, L, P, N = 400, 2, 1024, 3, 1500
    X, Y, w = _inputs(N, K, M, seed=31)
    m = _model(X, Y, w, folds=np.arange(N) % P)
    a = np.logspace(-3, 3, L) * _scale(m)
    rh = m.ridge_cross_validate(a, return_predictions=True)
    rd = m.ridge_cross_validate(a, return_predictions=True, out="torch")
    _same(rh, rd, RIDGE_KEYS + ("predictions", "rows"))
    for f in range(P):
        rf = m.ridge_cross_validate(a, fold_begin=f, fold_end=f + 1, return_predictions=True)
        assert np.array_equal(rf["predictions"], rh["predictions"][_span(m, f)]), f
    r1 = m.ridge_cross_validate(a, fold_begin=1, return_predictions=True, out="torch")
    assert np.array_equal(_np(r1["predictions"]), rh["predictions"][_span(m, 1).start:])
    sub = np.r_[0, 1, 511, 512, L - 1]
    _compare_ridge_pred(m, rh, X, a[sub], cols=sub)


def test_pls_staged_launches():
    # host predictions of A M = 2560 columns: the staging buffer holds `per` chunks, so PRESS of the range takes two
    # launches and fold 1 straddles their boundary; device outputs are written in one launch
    K, M, A = 64, 40, 64
    per = _stage_bytes() // (PRESS_ROWS * A * M * 8)
    n = PRESS_ROWS * (per // 2) + 40
    ch = -(-n // PRESS_ROWS)
    assert ch < per < 2 * ch < 2 * per
    X, Y, w = _inputs(2 * n, K, M, seed=64)
    m = _model(X, Y, w, folds=np.arange(2 * n) % 2)
    r0 = m.pls_cross_validate(A)
    rh = m.pls_cross_validate(A, return_predictions=True)
    rd = m.pls_cross_validate(A, return_predictions=True, out="torch")
    _same(r0, rh, PLS_KEYS)
    _same(rh, rd, PLS_KEYS + ("predictions", "rows"))
    r1 = m.pls_cross_validate(A, fold_begin=1, return_predictions=True)
    assert np.array_equal(r1["predictions"], rh["predictions"][n:])
    tb = m.training_batch()
    val = m._fold_indices[m._offsets[1]:m._offsets[2]]
    B, _ = po.ikpls(tb["XTX"][1], tb["XTY"][1], A)
    ref = po.predict(X[val], B, *_stats(m, tb, 1))
    assert _rel(rh["predictions"][n:, :8].transpose(1, 0, 2), ref[:8]) <= 1e-10


def test_ridge_staged_launches():
    # K = 4, M = 128, L = 1024: 32 MiB of float64 predictions per chunk, so a launch stages `per` chunks (fewer than the
    # plan's 255) and the two folds' chunks take two launches with fold 1 straddling the boundary
    K, M, L = 4, 128, 1024
    per = _stage_bytes() // (PRESS_ROWS * L * M * 8)
    n = PRESS_ROWS * (per // 2) + 22
    ch = -(-n // PRESS_ROWS)
    assert ch < per < 2 * ch
    X, Y, w = _inputs(2 * n, K, M, seed=404)
    m = _model(X, Y, w, folds=np.arange(2 * n) % 2)
    a = np.logspace(-3, 3, L) * _scale(m)
    r0 = m.ridge_cross_validate(a)
    rh = m.ridge_cross_validate(a, return_predictions=True)
    _same(r0, rh, RIDGE_KEYS)
    rd = m.ridge_cross_validate(a, return_predictions=True, out="torch")
    _same(rh, rd, RIDGE_KEYS + ("predictions", "rows"))
    del rd
    r1 = m.ridge_cross_validate(a, fold_begin=1, return_predictions=True)
    assert np.array_equal(r1["predictions"], rh["predictions"][n:])
    sub = np.r_[0, 511, L - 1]
    _compare_ridge_pred(m, {"predictions": rh["predictions"][:, sub]}, X, a[sub], cols=np.arange(3))
    _check_self_consistent(m, rh, X, Y, w)


# ---- 5. special rows -----------------------------------------------------------------------------------------------
def test_refused_fold_gives_nan_rows():
    X, Y, _ = _inputs(60, 6, 2, seed=3)
    w0 = np.zeros(60)
    w0[np.arange(60) % 3 == 1] = 1.0    # fold 1's training set has no non-zero weight
    m = _model(X, Y, w0, folds=np.arange(60) % 3)
    for out in ("numpy", "torch"):
        rp = m.pls_cross_validate(2, check=False, return_predictions=True, out=out)
        rr = m.ridge_cross_validate([0.1, 1.0], check=False, return_predictions=True, out=out)
        for r in (rp, rr):
            p = _np(r["predictions"])
            assert np.isnan(p[_span(m, 1)]).all()
            assert np.isfinite(p[_span(m, 0)]).all() and np.isfinite(p[_span(m, 2)]).all()


def test_failed_pair_is_nan_in_its_penalty_only():
    X, Y, w = _inputs(150, 20, 3, seed=6)
    X[:, 13] = 0.0
    m = _model(X, Y, w, flags=3, folds=np.arange(150) % 3)
    a = [0.0, 0.5, 0.0, 4.0]
    with pytest.warns(UserWarning):
        r = m.ridge_cross_validate(a, return_predictions=True)
    assert (r["info"][:, [0, 2]] == 14).all() and not r["info"][:, [1, 3]].any()
    assert np.isnan(r["predictions"][:, [0, 2]]).all() and np.isfinite(r["predictions"][:, [1, 3]]).all()
    _compare_ridge_pred(m, r, X, np.array(a))


def test_early_stop_repeats_last_component():
    rng = np.random.default_rng(2)
    X0 = rng.standard_normal((120, 3))
    X = np.hstack([X0, X0])
    Y = X0 @ rng.standard_normal((3, 2)) + 0.1 * rng.standard_normal((120, 2))
    m = _model(X, Y, None, folds=np.arange(120) % 3)
    with pytest.warns(UserWarning, match="stopped before 6 components"):
        r = m.pls_cross_validate(6, return_predictions=True)
    for f in range(3):
        nf = r["n_fitted"][f]
        p = r["predictions"][_span(m, f)]
        assert 1 <= nf < 6
        for a in range(nf, 6):
            assert np.array_equal(p[:, a], p[:, nf - 1])


def test_no_fitted_component_predicts_the_mean():
    # X = 0: XTY is exactly 0 in every fold (a constant Y with centring is not enough: the centred XTY of a fold keeps
    # rounding residue from the downdate, and a component is fitted on it), so no component is fitted and every
    # prediction is the fold's training mean of Y when Y is centred, else 0
    _, Y, _ = _inputs(90, 5, 2, seed=9)
    X = np.zeros((90, 5))
    for flags in (3, 1):
        m = _model(X, Y, None, flags=flags, folds=np.arange(90) % 3)
        with pytest.warns(UserWarning, match="stopped before 3 components"):
            r = m.pls_cross_validate(3, return_predictions=True)
        assert not r["n_fitted"].any() and not r["status"].any()
        tb = m.training_batch()
        for f in range(3):
            p = r["predictions"][_span(m, f)]
            mu = tb["Y_mean"][f].reshape(1, 1, 2) if flags & 2 else np.zeros((1, 1, 2))
            assert (flags & 2) == 0 or (mu != 0).all()
            assert np.array_equal(p, np.broadcast_to(mu, p.shape)), (flags, f)


def test_empty_folds_repeated_and_negative_indices():
    X, Y, w = _inputs(150, 9, 3, seed=8)
    rng = np.random.default_rng(1)
    sets = [np.arange(0, 40), np.array([], np.int64), np.array([5, 5, 7, -1, -1, 60]), rng.permutation(150)[:33],
            np.array([], np.int64), np.arange(100, 150)]
    m = _model(X, Y, w, sets=sets)
    a = np.array([0.1, 1.0, 10.0])
    for out in ("numpy", "torch"):
        for r in (m.pls_cross_validate(4, fold_begin=1, fold_end=5, return_predictions=True, out=out, return_coefs=True),
                  m.ridge_cross_validate(a, fold_begin=1, fold_end=5, return_predictions=True, out=out, return_coefs=True)):
            p = _np(r["predictions"])
            assert p.shape == (6 + 33, _np(r["press"]).shape[1], 3)
            _check_rows(m, r, 1, 5)
            rows = _np(r["rows"])
            assert rows[3] == 149 and rows[4] == 149
            assert np.array_equal(p[0], p[1]) and np.array_equal(p[3], p[4])
            if out == "numpy":
                _check_self_consistent(m, r, X, Y, w, 1, 5)
    for r in (m.pls_cross_validate(4, fold_begin=1, fold_end=2, return_predictions=True),
              m.ridge_cross_validate(a, fold_begin=4, fold_end=5, return_predictions=True, out="torch")):
        assert _np(r["predictions"]).shape[0] == 0 and _np(r["rows"]).shape == (0,)
    _compare_ridge_pred(m, m.ridge_cross_validate(a, return_predictions=True), X, a)


# ---- 6. end to end: scikit-learn's cross_val_predict ---------------------------------------------------------------
def test_pls_cross_val_predict_against_sklearn():
    from sklearn.cross_decomposition import PLSRegression

    X, Y, _ = _inputs(200, 12, 3, seed=8, weighted=False)
    P, A, N = 4, 4, 200
    folds = np.arange(N) % P
    m = _model(X, Y, None, folds=folds)
    r = m.pls_cross_validate(A, return_predictions=True)
    Yhat = np.empty((N, A, 3))
    Yhat[r["rows"]] = r["predictions"]
    for a in range(1, A + 1):
        ref = np.empty((N, 3))
        for f in range(P):
            val, train = folds == f, folds != f
            pls = PLSRegression(n_components=a, scale=True, tol=1e-30, max_iter=10000).fit(X[train], Y[train])
            ref[val] = pls.predict(X[val]).reshape(-1, 3)
        assert _rel(Yhat[:, a - 1], ref) <= 1e-9, a


def test_ridge_cross_val_predict_against_sklearn():
    from sklearn.linear_model import Ridge

    X, Y, w = _inputs(200, 12, 2, seed=7)
    w = w + 0.05
    P, N = 4, 200
    folds = np.arange(N) % P
    m = _model(X, Y, w, flags=3, folds=folds)
    alphas = [0.01, 1.0, 30.0, 1000.0]
    r = m.ridge_cross_validate(alphas, return_predictions=True)
    Yhat = np.empty((N, len(alphas), 2))
    Yhat[r["rows"]] = r["predictions"]
    for l, a in enumerate(alphas):
        ref = np.empty((N, 2))
        for f in range(P):
            val, train = folds == f, folds != f
            sk = Ridge(alpha=a, fit_intercept=True, solver="cholesky").fit(X[train], Y[train], sample_weight=w[train])
            ref[val] = sk.predict(X[val]).reshape(-1, 2)
        assert _rel(Yhat[:, l], ref) <= 1e-9, a


# ---- 7. streams and determinism ------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["float64", "float32"])
def test_torch_stream_and_determinism(dtype):
    import torch

    X, Y, w = _inputs(700, 40, 5, seed=9, dtype=dtype)
    m = _model(X, Y, w, dtype=dtype, folds=np.arange(700) % 7)
    a = np.logspace(-1, 1, 6) * _scale(m)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        p = [m.pls_cross_validate(8, out="torch", return_predictions=True) for _ in range(2)]
        q = [m.ridge_cross_validate(a, out="torch", return_predictions=True) for _ in range(2)]
        p = [{k: v.cpu().numpy() for k, v in d.items() if v is not None} for d in p]
        q = [{k: v.cpu().numpy() for k, v in d.items() if v is not None} for d in q]
    _same(p[0], p[1], PLS_KEYS + ("predictions", "rows"))
    _same(q[0], q[1], RIDGE_KEYS + ("predictions", "rows"))
    ph = m.pls_cross_validate(8, return_predictions=True)
    _same(ph, p[0], PLS_KEYS + ("predictions", "rows"))
