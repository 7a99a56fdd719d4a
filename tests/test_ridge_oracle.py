"""CPU tests of the cross-validated ridge oracle (oracle/ridge_oracle.py): against scikit-learn's Ridge with and without
an intercept, against least squares at lambda = 0, LAPACK's info convention on a singular matrix, and the
extended-precision solve (ridge_extended) against LAPACK."""

import numpy as np
import pytest

import ridge_oracle as ro


def _data(N, K, M, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, K)) + rng.standard_normal(K)
    Y = X @ rng.standard_normal((K, M)) + 0.3 * rng.standard_normal((N, M)) + 2.0
    w = rng.random(N) + 0.2
    return X, Y, w


@pytest.mark.parametrize("M", [1, 3])
def test_weighted_centred_matches_sklearn(M):
    from sklearn.linear_model import Ridge

    X, Y, w = _data(80, 6, M, seed=M)
    Xv, Yv, wv = _data(15, 6, M, seed=10 + M)
    # center_X | center_Y: weighted means, XTX = Xc^T W Xc, XTY = Xc^T W Yc
    mx, my = (w @ X) / w.sum(), (w @ Y) / w.sum()
    Xc, Yc = X - mx, Y - my
    XTX, XTY = Xc.T @ (w[:, None] * Xc), Xc.T @ (w[:, None] * Yc)
    alphas = [1e-3, 0.5, 7.0, 300.0]
    B, info = ro.ridge(XTX, XTY, alphas)
    assert not info.any()
    pr = ro.press(Xv, Yv, wv, B, *ro.fold_stats(3, mx, None, my, None))
    for l, a in enumerate(alphas):
        sk = Ridge(alpha=a, fit_intercept=True, solver="cholesky").fit(X, Y, sample_weight=w)
        np.testing.assert_allclose(B[l], sk.coef_.reshape(M, 6).T, rtol=1e-10, atol=1e-12)
        ref = wv @ ((Yv - sk.predict(Xv).reshape(-1, M)) ** 2)
        np.testing.assert_allclose(pr[l], ref, rtol=1e-10)


def test_no_flags_matches_sklearn_without_intercept():
    from sklearn.linear_model import Ridge

    X, Y, w = _data(60, 5, 2, seed=7)
    XTX, XTY = X.T @ (w[:, None] * X), X.T @ (w[:, None] * Y)
    B, info = ro.ridge(XTX, XTY, [0.1, 10.0])
    assert not info.any()
    for l, a in enumerate([0.1, 10.0]):
        sk = Ridge(alpha=a, fit_intercept=False, solver="cholesky").fit(X, Y, sample_weight=w)
        np.testing.assert_allclose(B[l], sk.coef_.T, rtol=1e-10, atol=1e-12)


def test_zero_penalty_is_least_squares():
    X, Y, w = _data(50, 7, 3, seed=3)
    sw = np.sqrt(w)[:, None]
    B, info = ro.ridge(X.T @ (w[:, None] * X), X.T @ (w[:, None] * Y), [0.0])
    ref = np.linalg.lstsq(sw * X, sw * Y, rcond=None)[0]
    assert info[0] == 0
    np.testing.assert_allclose(B[0], ref, rtol=1e-9, atol=1e-11)


@pytest.mark.parametrize("K,M", [(1, 1), (7, 3), (65, 2), (130, 5)])
def test_extended_matches_lapack(K, M):
    # well-conditioned systems: the float64 LAPACK solve and the extended one agree to a few kappa eps64
    X, Y, w = _data(3 * K + 20, K, M, seed=K)
    XTX, XTY = X.T @ (w[:, None] * X), X.T @ (w[:, None] * Y)
    alphas = [0.0, 0.1 * np.trace(XTX) / K, 10.0 * np.trace(XTX) / K]
    B, info = ro.ridge(XTX, XTY, alphas)
    Be, infoe = ro.ridge_extended(XTX, XTY, alphas)
    assert Be.dtype == np.longdouble and not info.any() and not infoe.any()
    ev = np.linalg.eigvalsh(XTX)
    for l, a in enumerate(alphas):
        kappa = (ev[-1] + a) / (ev[0] + a)
        err = np.linalg.norm((B[l] - Be[l]).astype(np.float64)) / np.linalg.norm(Be[l].astype(np.float64))
        assert err <= 5 * kappa * np.finfo(np.float64).eps, (l, err, kappa)
    # PRESS evaluated in extended precision from the extended B agrees with the float64 evaluation
    Xv, Yv, wv = _data(9, K, M, seed=100 + K)
    p64 = ro.press(Xv, Yv, wv, B)
    pe = ro.press(Xv, Yv, wv, Be, dtype=np.longdouble)
    assert pe.dtype == np.longdouble
    np.testing.assert_allclose(p64, pe.astype(np.float64), rtol=1e-9)


@pytest.mark.parametrize("j", [0, 37, 79])
def test_extended_info_matches_dpotrf(j):
    # an exactly zero column in the first, a middle and the last position: the same 1-based pivot as dpotrf
    X, Y, _ = _data(200, 80, 2, seed=j)
    X[:, j] = 0.0
    alphas = [0.0, 1.0, 0.0, 3.0]
    B, info = ro.ridge(X.T @ X, X.T @ Y, alphas)
    Be, infoe = ro.ridge_extended(X.T @ X, X.T @ Y, alphas)
    assert list(infoe) == list(info) == [j + 1, 0, j + 1, 0]
    assert np.isnan(Be[[0, 2]]).all() and np.isfinite(Be[[1, 3]]).all() and not Be[[1, 3]][:, j].any()
    assert np.abs((B[[1, 3]] - Be[[1, 3]]).astype(np.float64)).max() <= 1e-12 * np.abs(B[[1, 3]]).max()


def test_info_on_a_zero_column():
    X, Y, _ = _data(40, 6, 2, seed=5)
    X[:, 3] = 0.0
    B, info = ro.ridge(X.T @ X, X.T @ Y, [0.0, 1.0, 0.0])
    assert list(info) == [4, 0, 4]
    assert np.isnan(B[0]).all() and np.isnan(B[2]).all()
    assert np.isfinite(B[1]).all() and not B[1][3].any()
