"""CPU tests of the PLS cross-validation oracle (oracle/pls_oracle.py), the reference the GPU kernels of
CVMatrix.pls_cross_validate are checked against: IKPLS against scikit-learn's PLSRegression and least squares, the
early-stop rule, and the prediction rule for every flag combination."""

import itertools

import numpy as np
import pytest

import pls_oracle as po


def _standardise(A):
    mu, sd = A.mean(0), A.std(0, ddof=1)
    return (A - mu) / sd, mu, sd


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


@pytest.mark.parametrize("M", [1, 3])
@pytest.mark.parametrize("A", [1, 2, 5, 8])
def test_oracle_matches_sklearn(M, A):
    from sklearn.cross_decomposition import PLSRegression

    rng = np.random.default_rng(10 * M + A)
    N, K = 60, 8
    X = rng.standard_normal((N, K)) @ rng.standard_normal((K, K)) + rng.standard_normal(K)
    Y = X @ rng.standard_normal((K, M)) + 0.3 * rng.standard_normal((N, M)) + 2.0
    Xs, mx, sx = _standardise(X)
    Ys, my, sy = _standardise(Y)
    B, n_fitted = po.ikpls(Xs.T @ Xs, Xs.T @ Ys, A)
    assert n_fitted == A
    ref = PLSRegression(n_components=A, scale=True, tol=1e-30, max_iter=10000).fit(X, Y).predict(X).reshape(N, M)
    got = po.predict(X, B, mx, sx, my, sy)[A - 1]
    assert _rel(got, ref) <= 1e-12
    # fewer components: the leading coefficients of the same fit
    for a in range(1, A):
        ref_a = PLSRegression(n_components=a, scale=True, tol=1e-30, max_iter=10000).fit(X, Y).predict(X).reshape(N, M)
        assert _rel(po.predict(X, B, mx, sx, my, sy)[a - 1], ref_a) <= 1e-12


@pytest.mark.parametrize("M", [1, 3])
def test_all_components_equal_least_squares(M):
    rng = np.random.default_rng(7)
    N, K = 50, 6
    X, Y = rng.standard_normal((N, K)), rng.standard_normal((N, M))
    Xs, _, _ = _standardise(X)
    Ys, _, _ = _standardise(Y)
    B, n_fitted = po.ikpls(Xs.T @ Xs, Xs.T @ Ys, K)
    assert n_fitted == K
    ls = np.linalg.lstsq(Xs, Ys, rcond=None)[0]
    assert _rel(B[-1], ls) <= 1e-12


@pytest.mark.parametrize("M", [1, 2])
def test_early_stop_on_rank_deficient_X(M):
    rng = np.random.default_rng(3)
    N = 40
    X0 = rng.standard_normal((N, 3))
    X = np.hstack([X0, X0])           # rank 3 with K = 6
    Y = rng.standard_normal((N, M))
    Xs, _, _ = _standardise(X)
    Ys, _, _ = _standardise(Y)
    A = 6
    B, n_fitted = po.ikpls(Xs.T @ Xs, Xs.T @ Ys, A)
    assert 1 <= n_fitted < A
    for a in range(n_fitted, A):
        assert np.array_equal(B[a], B[n_fitted - 1])
    # nothing to fit at all: B stays zero
    B0, n0 = po.ikpls(Xs.T @ Xs, np.zeros((6, M)), 3)
    assert n0 == 0 and not B0.any()


@pytest.mark.parametrize("flags", range(16))
def test_prediction_rule_all_flags(flags):
    rng = np.random.default_rng(flags)
    n, K, M, A = 7, 5, 3, 4
    Xv, Yv, w = rng.standard_normal((n, K)), rng.standard_normal((n, M)), rng.random(n)
    B = rng.standard_normal((A, K, M))
    mx, sx, my, sy = rng.standard_normal(K), rng.random(K) + 0.5, rng.standard_normal(M), rng.random(M) + 0.5
    stats = po.fold_stats(flags, mx, sx, my, sy)
    got = po.predict(Xv, B, *stats)
    got_press = po.press(Xv, Yv, w, B, *stats)
    for a, i in itertools.product(range(A), range(n)):
        x = Xv[i].copy()
        if flags & 1:
            x = x - mx
        if flags & 4:
            x = x / sx
        y = x @ B[a]
        if flags & 8:
            y = y * sy
        if flags & 2:
            y = y + my
        np.testing.assert_allclose(got[a, i], y, rtol=1e-14, atol=1e-14)
    direct = np.array([[sum(w[i] * (Yv[i, m] - got[a, i, m]) ** 2 for i in range(n)) for m in range(M)] for a in range(A)])
    np.testing.assert_allclose(got_press, direct, rtol=1e-13)
