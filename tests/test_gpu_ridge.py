"""
GPU tests (-m gpu) of cross-validated ridge regression (cvmx_ridge_cv / CVMatrix.ridge_cross_validate): the kernels
against the LAPACK oracle fed with the engine's own training matrices, end to end against scikit-learn, exact
properties of singular folds and huge penalties, fold shapes, windows and passes, the fold-Gram cache, streams and
determinism, and the argument / degenerate-fold errors.  Ordered from small shapes to large.
"""

import warnings

import numpy as np
import pytest

import ridge_oracle as ro
from cvmatrix_oracle import ERR_NO_NONZERO

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


def _inputs(N, K, M, seed, weighted=True, dtype=np.float64):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, K)) + rng.standard_normal(K)
    Y = X @ rng.standard_normal((K, M)) / np.sqrt(K) + 0.5 * rng.standard_normal((N, M)) + 1.0
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


def _alphas(m, L, lo=1e-3, hi=1e3):
    """Penalties spread over lo .. hi times trace(XTX) / K of the first fold."""
    XTX = m.training_batch(0, 1)["XTX"][0].astype(np.float64)
    return np.logspace(np.log10(lo), np.log10(hi), L) * np.trace(XTX) / XTX.shape[0]


def _oracle(m, X, Y, w, alphas, f0=0, f1=None):
    """Oracle ridge + PRESS on the engine's own training matrices and statistics (isolates the ridge kernels)."""
    f1 = m._n_folds if f1 is None else f1
    tb = m.training_batch(f0, f1, check=False)
    X64, Y64 = X.astype(np.float64), Y.astype(np.float64)
    out = []
    for i in range(f1 - f0):
        f = f0 + i
        val = m._fold_indices[m._offsets[f]:m._offsets[f + 1]]
        XTX = tb["XTX"][i].astype(np.float64)
        B, info = ro.ridge(XTX, tb["XTY"][i], alphas)
        g = lambda k: None if tb[k] is None else tb[k][i].astype(np.float64)  # noqa: E731
        stats = ro.fold_stats(m._flags, g("X_mean"), g("X_std"), g("Y_mean"), g("Y_std"))
        wv = None if w is None else w[val].astype(np.float64)
        kappa = np.array([np.linalg.cond(XTX + a * np.eye(len(XTX))) for a in alphas])
        out.append((B, info, ro.press(X64[val], Y64[val], wv, B, *stats), len(val) if w is None else wv.sum(), kappa))
    return out


def _rel(a, b):
    nb = np.linalg.norm(b)
    return np.linalg.norm(a - b) / (nb if nb > 0 else 1.0)


def _compare(r, ref, f0=0, check_B=True, extra=0.0):
    """info exactly; B and press to 50 kappa eps (kappa: 2-norm condition number of XTX + lambda I), plus `extra` for
    outputs rounded to float32."""
    for i, (B, info, pr, sw, kappa) in enumerate(ref):
        assert np.array_equal(r["info"][f0 + i], info), (f0 + i, r["info"][f0 + i], info)
        assert abs(float(r["sum_w_val"][f0 + i]) - sw) <= 1e-6 * max(sw, 1.0)
        for l in range(len(info)):
            if info[l]:
                assert np.isnan(r["press"][f0 + i, l]).all()
                continue
            tol = 50.0 * kappa[l] * EPS + extra
            assert _rel(r["press"][f0 + i, l].astype(np.float64), pr[l]) <= tol, (f0 + i, l, _rel(r["press"][f0 + i, l], pr[l]), tol)
            if check_B:
                assert _rel(r["B"][f0 + i, l].astype(np.float64), B[l]) <= tol, (f0 + i, l, _rel(r["B"][f0 + i, l], B[l]), tol)


def test_tiny_single_panel():
    X, Y, w = _inputs(60, 5, 2, seed=1)
    m = _model(X, Y, w, folds=np.arange(60) % 3)
    a = _alphas(m, 4)
    r = m.ridge_cross_validate(a, return_coefs=True)
    assert r["press"].shape == (3, 4, 2) and r["B"].shape == (3, 4, 5, 2) and r["info"].shape == (3, 4)
    assert r["info"].dtype == np.int32 and not r["status"].any()
    _compare(r, _oracle(m, X, Y, w, a))


@pytest.mark.parametrize("K", [64, 300])
@pytest.mark.parametrize("M", [1, 3, 40])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_kernel_parity(K, M, dtype):
    X, Y, w = _inputs(900, K, M, seed=K + M, dtype=dtype)
    P = 5
    m = _model(X, Y, w, dtype=dtype, folds=np.arange(900) % P)
    a = _alphas(m, 7)
    r = m.ridge_cross_validate(a, return_coefs=True)
    assert r["press"].shape == (P, 7, M) and r["B"].shape == (P, 7, K, M) and r["press"].dtype == dtype
    if dtype == np.float64:
        _compare(r, _oracle(m, X, Y, w, a))
    else:   # float64 arithmetic, outputs rounded to float32
        _compare(r, _oracle(m, X, Y, w, a), extra=1e-6)


@pytest.mark.parametrize("flags", range(16))
def test_all_flag_combinations(flags):
    X, Y, w = _inputs(120, 10, 2, seed=100 + flags)
    m = _model(X, Y, w, flags=flags, folds=np.arange(120) % 4)
    a = _alphas(m, 3)
    r = m.ridge_cross_validate(a, return_coefs=True)
    _compare(r, _oracle(m, X, Y, w, a))


@pytest.mark.parametrize("M", [1, 3])
def test_end_to_end_against_sklearn(M):
    from sklearn.linear_model import Ridge

    X, Y, w = _inputs(200, 12, M, seed=5 + M)
    w = w + 0.05
    P = 4
    folds = np.arange(200) % P
    m = _model(X, Y, w, flags=3, folds=folds)   # center_X | center_Y: Ridge(fit_intercept=True)
    alphas = [0.01, 1.0, 30.0, 1000.0]
    r = m.ridge_cross_validate(alphas, return_coefs=True)
    for f in range(P):
        val, train = folds == f, folds != f
        for l, a in enumerate(alphas):
            sk = Ridge(alpha=a, fit_intercept=True, solver="cholesky").fit(X[train], Y[train], sample_weight=w[train])
            ref = w[val] @ ((Y[val] - sk.predict(X[val]).reshape(-1, M)) ** 2)
            assert _rel(r["press"][f, l], ref) <= 1e-9
            assert _rel(r["B"][f, l], sk.coef_.reshape(M, 12).T) <= 1e-9
        assert abs(r["sum_w_val"][f] - w[val].sum()) <= 1e-12 * w[val].sum()


def test_zero_column_info_and_exact_zero_row():
    X, Y, w = _inputs(150, 20, 3, seed=6)
    j = 13
    X[:, j] = 0.0
    m = _model(X, Y, w, flags=3, folds=np.arange(150) % 3)   # no scaling: the zero column stays exactly zero
    alphas = [0.0, 0.5, 0.0, 4.0]
    with pytest.warns(UserWarning, match="6 \\(fold, penalty\\) pair"):
        r = m.ridge_cross_validate(alphas, return_coefs=True)
    assert (r["info"][:, [0, 2]] == j + 1).all() and not r["info"][:, [1, 3]].any()
    assert np.isnan(r["press"][:, [0, 2]]).all() and np.isnan(r["B"][:, [0, 2]]).all()
    assert np.isfinite(r["press"][:, [1, 3]]).all() and np.isfinite(r["B"][:, [1, 3]]).all()
    assert (r["B"][:, [1, 3], j, :] == 0).all()
    _compare(r, _oracle(m, X, Y, w, alphas))


def test_huge_penalty_is_intercept_only():
    X, Y, w = _inputs(200, 15, 2, seed=12)
    folds = np.arange(200) % 4
    for flags in (2, 3, 15):
        m = _model(X, Y, w, flags=flags, folds=folds)
        tb = m.training_batch()
        a = 1e12 * np.trace(tb["XTX"][0])
        r = m.ridge_cross_validate([a])
        for f in range(4):
            val = folds == f
            ref = w[val] @ ((Y[val] - tb["Y_mean"][f]) ** 2)
            assert _rel(r["press"][f, 0], ref) <= 1e-9, flags


def test_leave_one_out_and_leave_few_out():
    X, Y, w = _inputs(90, 8, 2, seed=21)
    for folds in (np.arange(90), np.arange(90) // 3):
        m = _model(X, Y, w, folds=folds)
        a = _alphas(m, 5)
        r = m.ridge_cross_validate(a, return_coefs=True)
        _compare(r, _oracle(m, X, Y, w, a))


def test_range_empty_fold_repeated_and_negative_indices():
    X, Y, w = _inputs(150, 9, 3, seed=8)
    rng = np.random.default_rng(1)
    sets = [np.arange(0, 40), np.array([], np.int64), np.array([5, 5, 7, -1, -1, 60]), rng.permutation(150)[:33],
            np.arange(100, 150)]
    m = _model(X, Y, w, sets=sets)
    a = _alphas(m, 4)
    r = m.ridge_cross_validate(a, fold_begin=1, fold_end=5, return_coefs=True)
    assert r["press"].shape == (4, 4, 3)
    _compare(r, _oracle(m, X, Y, w, a, 1, 5))
    assert not r["press"][0].any() and r["sum_w_val"][0] == 0     # the empty fold
    full = m.ridge_cross_validate(a)
    assert _rel(full["press"][1:], r["press"]) <= 1e-12
    empty = m.ridge_cross_validate(a, fold_begin=2, fold_end=2)
    assert empty["press"].shape == (0, 4, 3) and empty["info"].shape == (0, 4)


def test_torch_stream_and_determinism():
    import torch

    X, Y, w = _inputs(700, 70, 5, seed=9)
    m = _model(X, Y, w, folds=np.arange(700) % 7)
    a = np.concatenate([_alphas(m, 6), [0.0, 3.0, 3.0]])   # repeats allowed
    r1 = m.ridge_cross_validate(a, return_coefs=True)
    r2 = m.ridge_cross_validate(a, return_coefs=True)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        rt = m.ridge_cross_validate(torch.tensor(a), return_coefs=True, out="torch")
        assert rt["press"].is_cuda and rt["B"].is_cuda and rt["info"].is_cuda
        rt = {k: v.cpu().numpy() for k, v in rt.items()}
    for k in ("press", "sum_w_val", "info", "status", "B"):
        assert np.array_equal(r1[k], r2[k]) and np.array_equal(r1[k], rt[k]), k
    assert np.array_equal(r1["press"][:, 7], r1["press"][:, 8])


def test_fold_gram_cache():
    from cvmatrix_b200 import CVMatrix, Partitioner

    X, Y, w = _inputs(450_000, 48, 3, seed=4)    # large enough for the chunk-pipelined upload that keeps fold Grams
    part = Partitioner(np.arange(450_000) % 5)
    a = CVMatrix(copy=False)
    a.fit(X, Y, w, folds=part)
    assert a.folds_cached
    alphas = _alphas(a, 5)
    ra = a.ridge_cross_validate(alphas, return_coefs=True)
    assert a.folds_cached
    b = CVMatrix(copy=False)
    b.fit(X, Y, w)
    b.set_folds(part)
    rb = b.ridge_cross_validate(alphas, return_coefs=True)
    assert np.array_equal(ra["info"], rb["info"])
    assert _rel(ra["press"], rb["press"]) <= 1e-9 and _rel(ra["B"], rb["B"]) <= 1e-9


def test_errors_and_unchecked_status():
    from cvmatrix_b200 import CVMatrix, Partitioner

    X, Y, w = _inputs(60, 6, 2, seed=3)
    m = _model(X, Y, w, folds=np.arange(60) % 3)
    for bad in ([], [[1.0, 2.0]], [1.0, -1.0], [np.nan], [np.inf], np.ones(1025), "abc"):
        with pytest.raises(ValueError, match="alphas|penalt"):
            m.ridge_cross_validate(bad)
    wide = CVMatrix()
    wide.fit(X, np.zeros((60, 129)) + np.arange(129))
    wide.set_folds(Partitioner(np.arange(60) % 3))
    with pytest.raises(ValueError, match="128"):
        wide.ridge_cross_validate([1.0])
    noy = CVMatrix()
    noy.fit(X)
    noy.set_folds(Partitioner(np.arange(60) % 3))
    with pytest.raises(ValueError, match="Response variables `Y` are not provided."):
        noy.ridge_cross_validate([1.0])
    # every non-zero weight sits in fold 1's validation rows: its training set has none
    w0 = np.zeros(60)
    w0[np.arange(60) % 3 == 1] = 1.0
    z = _model(X, Y, w0, folds=np.arange(60) % 3)
    with pytest.raises(ValueError, match=ERR_NO_NONZERO):
        z.ridge_cross_validate([1.0, 2.0])
    with warnings.catch_warnings():
        warnings.simplefilter("error")     # a refused fold is reported through status, not as a failed factorisation
        r = z.ridge_cross_validate([1.0, 2.0], check=False, return_coefs=True)
    assert r["status"][1] & 1 and not r["info"][1].any()
    assert np.isnan(r["press"][1]).all() and np.isnan(r["B"][1]).all()
    assert not r["status"][0] and np.isfinite(r["press"][0]).all() and np.isfinite(r["B"][0]).all()


def test_range_spanning_windows_and_passes():
    # K = 400, L = 1024: one fold with all penalties exceeds the ~1 GiB pass, so every fold is its own window and its
    # penalties go in several passes (test_ridge_plan.py checks the plan of this shape)
    import ctypes as C

    from cvmatrix_b200 import _lib

    K, M, L, P = 400, 2, 1024, 3
    plan = np.zeros(_lib.RIDGE_PLAN_LEN, np.int64)
    assert _lib.load().cvmx_ridge_plan(K, M, L, P, 1, 0, 0, plan.ctypes.data_as(C.c_void_p)) == 0
    W, Lp = plan[_lib.RIDGE_FOLDS_PER_WINDOW], plan[_lib.RIDGE_PENALTIES_PER_PASS]
    assert W < P and Lp < L
    X, Y, w = _inputs(1500, K, M, seed=31)
    m = _model(X, Y, w, folds=np.arange(1500) % P)
    a = _alphas(m, L)
    r = m.ridge_cross_validate(a)
    sub = np.r_[0:3, Lp - 2:Lp + 2, L - 3:L]   # penalties on both sides of a pass boundary
    ref = _oracle(m, X, Y, w, a[sub])
    _compare({"press": r["press"][:, sub], "info": r["info"][:, sub], "sum_w_val": r["sum_w_val"]}, ref, check_B=False)
    for f0, f1 in ((0, 1), (1, 3), (2, 3)):
        rs = m.ridge_cross_validate(a, fold_begin=f0, fold_end=f1)
        assert _rel(rs["press"], r["press"][f0:f1]) <= 1e-12 and np.array_equal(rs["info"], r["info"][f0:f1])
