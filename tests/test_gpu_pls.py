"""
GPU tests (-m gpu) of cross-validated PLS (cvmx_pls_cv / CVMatrix.pls_cross_validate): the kernels against the numpy
IKPLS oracle fed with the engine's own training matrices, end to end against scikit-learn, fold shapes, the fold-Gram
cache, streams and determinism, and the argument / degenerate-fold errors.
"""

import warnings

import numpy as np
import pytest

import pls_oracle as po
from cvmatrix_oracle import ERR_NO_NONZERO

pytestmark = pytest.mark.gpu

FLAGS_ALL = 15


def _inputs(N, K, M, seed, weighted=True, dtype=np.float64):
    """Responses with a planted linear signal (well separated PLS directions) plus noise; some zero weights."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, K)) + rng.standard_normal(K)
    C = rng.standard_normal((K, M)) * (0.8 ** np.arange(M))
    Y = X @ C / np.sqrt(K) + 0.5 * rng.standard_normal((N, M)) + 1.0
    w = None
    if weighted:
        w = rng.random(N) + 0.1
        w[::7] = 0.0
    return X.astype(dtype), Y.astype(dtype), (None if w is None else w.astype(dtype))


def _model(X, Y, w, flags=FLAGS_ALL, dtype=np.float64, folds=None, sets=None):
    from cvmatrix_b200 import CVMatrix, Partitioner

    m = CVMatrix(center_X=bool(flags & 1), center_Y=bool(flags & 2), scale_X=bool(flags & 4), scale_Y=bool(flags & 8),
                 dtype=dtype)
    m.fit(X, Y, w)
    if sets is not None:
        m.set_folds(sets)
    else:
        m.set_folds(Partitioner(folds))
    return m


def _oracle(m, X, Y, w, A, f0=0, f1=None):
    """Oracle IKPLS + PRESS on the engine's own training matrices and statistics (isolates the PLS kernels)."""
    f1 = m._n_folds if f1 is None else f1
    tb = m.training_batch(f0, f1)
    flags = m._flags
    X64, Y64 = X.astype(np.float64), Y.astype(np.float64)
    out = []
    for i in range(f1 - f0):
        f = f0 + i
        val = m._fold_indices[m._offsets[f]:m._offsets[f + 1]]
        B, nf = po.ikpls(tb["XTX"][i], tb["XTY"][i], A)
        g = lambda k: None if tb[k] is None else tb[k][i].astype(np.float64)  # noqa: E731
        stats = po.fold_stats(flags, g("X_mean"), g("X_std"), g("Y_mean"), g("Y_std"))
        wv = None if w is None else w[val].astype(np.float64)
        out.append((B, nf, po.press(X64[val], Y64[val], wv, B, *stats), len(val) if w is None else wv.sum()))
    return out


def _rel(a, b):
    nb = np.linalg.norm(b)
    return np.linalg.norm(a - b) / (nb if nb > 0 else 1.0)


def _compare(r, ref, tol_b, tol_p, f0=0, check_B=True):
    for i, (B, nf, pr, sw) in enumerate(ref):
        assert r["n_fitted"][f0 + i] == nf, (f0 + i, r["n_fitted"][f0 + i], nf)
        assert _rel(r["press"][f0 + i].astype(np.float64), pr) <= tol_p, (f0 + i, _rel(r["press"][f0 + i], pr))
        assert abs(float(r["sum_w_val"][f0 + i]) - sw) <= 1e-6 * max(sw, 1.0)
        if check_B:
            for a in range(B.shape[0]):
                assert _rel(r["B"][f0 + i, a].astype(np.float64), B[a]) <= tol_b, (f0 + i, a)


@pytest.mark.parametrize("K", [64, 300])
@pytest.mark.parametrize("M", [1, 3, 40])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_kernel_parity(K, M, dtype):
    X, Y, w = _inputs(900, K, M, seed=K + M, dtype=dtype)
    P, A = 5, 15
    m = _model(X, Y, w, dtype=dtype, folds=np.arange(900) % P)
    r = m.pls_cross_validate(A, return_coefs=True)
    assert r["press"].shape == (P, A, M) and r["B"].shape == (P, A, K, M) and r["press"].dtype == dtype
    assert r["n_fitted"].dtype == np.int32 and not r["status"].any()
    tol = (1e-10, 1e-9) if dtype == np.float64 else (2e-5, 2e-5)
    _compare(r, _oracle(m, X, Y, w, A), *tol)


@pytest.mark.parametrize("flags", range(16))
def test_all_flag_combinations(flags):
    X, Y, w = _inputs(120, 10, 2, seed=100 + flags)
    m = _model(X, Y, w, flags=flags, folds=np.arange(120) % 4)
    r = m.pls_cross_validate(5, return_coefs=True)
    _compare(r, _oracle(m, X, Y, w, 5), 1e-10, 1e-9)


@pytest.mark.parametrize("M", [1, 3])
def test_end_to_end_against_sklearn(M):
    from sklearn.cross_decomposition import PLSRegression

    X, Y, _ = _inputs(200, 12, M, seed=5 + M, weighted=False)
    P, A = 4, 4
    folds = np.arange(200) % P
    m = _model(X, Y, None, folds=folds)
    r = m.pls_cross_validate(A)
    for f in range(P):
        val, train = folds == f, folds != f
        for a in range(1, A + 1):
            pls = PLSRegression(n_components=a, scale=True, tol=1e-30, max_iter=10000).fit(X[train], Y[train])
            ref = ((Y[val] - pls.predict(X[val]).reshape(-1, M)) ** 2).sum(0)
            assert _rel(r["press"][f, a - 1], ref) <= 1e-9
        assert r["sum_w_val"][f] == val.sum()


def test_leave_one_out_and_leave_few_out():
    X, Y, w = _inputs(90, 8, 2, seed=21)
    for folds in (np.arange(90), np.arange(90) // 3):
        m = _model(X, Y, w, folds=folds)
        r = m.pls_cross_validate(6, return_coefs=True)
        _compare(r, _oracle(m, X, Y, w, 6), 1e-10, 1e-9)


def test_range_empty_fold_repeated_and_negative_indices():
    X, Y, w = _inputs(150, 9, 3, seed=8)
    rng = np.random.default_rng(1)
    sets = [np.arange(0, 40), np.array([], np.int64), np.array([5, 5, 7, -1, -1, 60]), rng.permutation(150)[:33],
            np.arange(100, 150)]
    m = _model(X, Y, w, sets=sets)
    r = m.pls_cross_validate(4, fold_begin=1, fold_end=5, return_coefs=True)
    assert r["press"].shape == (4, 4, 3)
    _compare(r, _oracle(m, X, Y, w, 4, 1, 5), 1e-10, 1e-9, f0=0)
    assert not r["press"][0].any() and r["sum_w_val"][0] == 0     # the empty fold
    full = m.pls_cross_validate(4)
    assert _rel(full["press"][1:], r["press"]) <= 1e-12 and np.array_equal(full["n_fitted"][1:], r["n_fitted"])


def test_range_spanning_staging_windows():
    # leave-one-out, K = 256: about 0.6 MB of device scratch per fold, so 2500 folds take two ~1 GiB windows
    X, Y, w = _inputs(2500, 256, 2, seed=77)
    m = _model(X, Y, w, folds=np.arange(2500))
    r = m.pls_cross_validate(4)
    for f0, f1 in ((0, 20), (1150, 1250), (1900, 2000), (2480, 2500)):   # the first window ends near fold 1945
        ref = _oracle(m, X, Y, w, 4, f0, f1)
        _compare(r, ref, 0, 1e-9, f0=f0, check_B=False)


def test_fold_gram_cache():
    from cvmatrix_b200 import CVMatrix, Partitioner

    X, Y, w = _inputs(450_000, 48, 3, seed=4)    # large enough for the chunk-pipelined upload that keeps fold Grams
    part = Partitioner(np.arange(450_000) % 5)
    a = CVMatrix(copy=False)
    a.fit(X, Y, w, folds=part)
    assert a.folds_cached
    ra = a.pls_cross_validate(6, return_coefs=True)
    assert a.folds_cached
    b = CVMatrix(copy=False)
    b.fit(X, Y, w)
    b.set_folds(part)
    rb = b.pls_cross_validate(6, return_coefs=True)
    assert np.array_equal(ra["n_fitted"], rb["n_fitted"])
    assert _rel(ra["press"], rb["press"]) <= 1e-9 and _rel(ra["B"], rb["B"]) <= 1e-9


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_torch_stream_and_determinism(dtype):
    import torch

    X, Y, w = _inputs(700, 40, 5, seed=9, dtype=dtype)
    m = _model(X, Y, w, dtype=dtype, folds=np.arange(700) % 7)
    r1 = m.pls_cross_validate(8, return_coefs=True)
    r2 = m.pls_cross_validate(8, return_coefs=True)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        rt = m.pls_cross_validate(8, return_coefs=True, out="torch")
        assert rt["press"].is_cuda and rt["B"].is_cuda
        rt = {k: v.cpu().numpy() for k, v in rt.items()}
    for k in ("press", "sum_w_val", "n_fitted", "status", "B"):
        assert np.array_equal(r1[k], r2[k]) and np.array_equal(r1[k], rt[k]), k


def test_early_stop_on_rank_deficient_X():
    rng = np.random.default_rng(2)
    X0 = rng.standard_normal((120, 3))
    X = np.hstack([X0, X0])
    Y = X0 @ rng.standard_normal((3, 2)) + 0.1 * rng.standard_normal((120, 2))
    m = _model(X, Y, None, folds=np.arange(120) % 3)
    with pytest.warns(UserWarning, match="stopped before 6 components"):
        r = m.pls_cross_validate(6, return_coefs=True)
    for f in range(3):
        nf = r["n_fitted"][f]
        assert 1 <= nf < 6
        for a in range(nf, 6):
            assert np.array_equal(r["B"][f, a], r["B"][f, nf - 1])
            assert np.array_equal(r["press"][f, a], r["press"][f, nf - 1])


def test_errors_and_unchecked_status():
    from cvmatrix_b200 import CVMatrix, Partitioner

    X, Y, w = _inputs(60, 6, 2, seed=3)
    m = _model(X, Y, w, folds=np.arange(60) % 3)
    for A in (0, 7):
        with pytest.raises(ValueError, match="n_components"):
            m.pls_cross_validate(A)
    wide = CVMatrix()
    wide.fit(X, np.zeros((60, 129)) + np.arange(129))
    wide.set_folds(Partitioner(np.arange(60) % 3))
    with pytest.raises(ValueError, match="128"):
        wide.pls_cross_validate(2)
    noy = CVMatrix()
    noy.fit(X)
    noy.set_folds(Partitioner(np.arange(60) % 3))
    with pytest.raises(ValueError, match="Response variables `Y` are not provided."):
        noy.pls_cross_validate(2)
    # every non-zero weight sits in fold 1's validation rows: its training set has none
    w0 = np.zeros(60)
    w0[np.arange(60) % 3 == 1] = 1.0
    z = _model(X, Y, w0, folds=np.arange(60) % 3)
    with pytest.raises(ValueError, match=ERR_NO_NONZERO):
        z.pls_cross_validate(2)
    with warnings.catch_warnings():
        warnings.simplefilter("error")     # a refused fold is reported through status, not as an early stop
        r = z.pls_cross_validate(2, check=False, return_coefs=True)
    assert r["status"][1] & 1 and r["n_fitted"][1] == 0
    assert np.isnan(r["press"][1]).all() and np.isnan(r["B"][1]).all()
    assert not r["status"][0] and np.isfinite(r["press"][0]).all()
