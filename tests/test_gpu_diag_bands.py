"""
GPU tests (-m gpu) of the band assignment of diagonal Gram tiles (kernels_gram.cuh, GDIAG_MASK): a diagonal tile
computes only its 16 x 16 bands on or above the diagonal, two warps compute bands of another warp's tile and hand
them over through shared memory.  Every K from 2 to 500 around the 16-row band and 128-column tile edges, with and
without Y, through each path that consumes the fragments: single-unit folds (fused statistics unless M = 1),
row-split folds (partials + k_gram_reduce), XTX-only and XTY-only batches, the fit totals, the streaming fit, the
fused fit + folds and float32 on k_gram<float>.  Matrices against the oracle at the bars of the other suites, XTX
exactly symmetric, statistics bit for bit.
"""

import os

import numpy as np
import pytest

from cvmatrix_oracle import OracleCVMatrix, make_inputs, rel_fro

pytestmark = pytest.mark.gpu

KS = [2, 9, 15, 16, 17, 31, 33, 63, 65, 127, 128, 129, 255, 257, 500]
STATS = ("X_mean", "X_std", "Y_mean", "Y_std")


def _inputs(N, K, M, seed, dtype=np.float64):
    X, Y, w, _ = make_inputs(N, K, max(M, 1), 1, dtype=dtype, seed=seed)
    w[::13] = 0
    return X, (Y if M else None), w


def _check_fold(out, pos, r, has_Y, want_XTX=True, want_XTY=True):
    if want_XTX:
        XTX = out["XTX"][pos]
        assert np.array_equal(XTX, XTX.T)
        assert rel_fro(XTX, r.XTX) <= 1e-12
    if has_Y and want_XTY:
        assert rel_fro(out["XTY"][pos], r.XTY) <= 6e-12
        if want_XTX:
            assert rel_fro(np.hstack([out["XTX"][pos], out["XTY"][pos]]), np.hstack([r.XTX, r.XTY])) <= 1e-12
    for s in STATS:
        got, exp = out.get(s), getattr(r, s)
        if got is not None and exp is not None:
            assert np.array_equal(got[pos], exp), s


@pytest.mark.parametrize("M", [0, 1, 10, 130])
@pytest.mark.parametrize("K", KS)
def test_diagonal_bands_fold_paths(K, M):
    from cvmatrix_b200 import CVMatrix, Partitioner

    N = 12_000
    X, Y, w = _inputs(N, K, M, seed=K * 7 + M)
    has_Y = Y is not None
    m = CVMatrix()
    m.fit(X, Y, w)
    orc = OracleCVMatrix()
    orc.fit(X, Y, w)
    assert np.array_equal(m.XTX, m.XTX.T) and rel_fro(m.XTX, orc.XTX) <= 1e-12
    if has_Y:
        assert rel_fro(m.XTY, orc.XTY) <= 1e-12
    # two folds of 6000 rows: row-split units, partials summed by k_gram_reduce
    # sixty folds of 200 rows: one unit per fold, epilogue (and, with M != 1, the statistics) inside k_gram
    for P, picks in ((2, (0, 1)), (60, (0, 31, 59))):
        folds = np.arange(N) % P
        m.set_folds(Partitioner(folds))
        out = m.training_batch(return_XTY=has_Y)
        for pos in picks:
            r = orc.fold(np.flatnonzero(folds == pos), want_XTY=has_Y)
            _check_fold(out, pos, r, has_Y)
            assert out["sum_w_train"][pos] == r.sum_w_train and out["nnz_train"][pos] == r.nnz_train
        if P == 60:
            xx = m.training_batch(return_XTY=False)
            for pos in picks:
                _check_fold(xx, pos, orc.fold(np.flatnonzero(folds == pos), want_XTY=False), has_Y, want_XTY=False)
                assert np.array_equal(xx["X_std"][pos], out["X_std"][pos])
            if has_Y:
                xy = m.training_batch(return_XTX=False)
                for pos in picks:
                    _check_fold(xy, pos, orc.fold(np.flatnonzero(folds == pos)), has_Y, want_XTX=False)


@pytest.mark.parametrize("K", KS)
def test_diagonal_bands_streaming_fit(K):
    from cvmatrix_b200 import CVMatrix, Partitioner

    N, M = 9_000, 10
    X, Y, w = _inputs(N, K, M, seed=K + 101)
    m = CVMatrix()
    m.fit_begin(N, K, M, weighted=True, max_block_rows=4_000)
    for r0 in (4_000, 0, 8_000):   # out of order, uneven
        r1 = min(N, r0 + 4_000)
        m.fit_rows(r0, X[r0:r1], Y[r0:r1], w[r0:r1])
    m.fit_end()
    orc = OracleCVMatrix()
    orc.fit(X, Y, w)
    assert np.array_equal(m.XTX, m.XTX.T) and rel_fro(m.XTX, orc.XTX) <= 1e-12 and rel_fro(m.XTY, orc.XTY) <= 1e-12
    folds = np.arange(N) % 3
    m.set_folds(Partitioner(folds))
    out = m.training_batch()
    _check_fold(out, 1, orc.fold(np.flatnonzero(folds == 1)), True)


@pytest.mark.parametrize("K", [17, 129, 257])
def test_diagonal_bands_fused_fit_folds(K):
    from cvmatrix_b200 import CVMatrix, Partitioner

    N, M, P = 12_000_000 // K, 10, 4      # 96 MB of X: the chunked upload, where fit(..., folds=) keeps the fold Grams
    X, Y, w = _inputs(N, K, M, seed=K + 202)
    part = Partitioner(np.arange(N) % P)
    m = CVMatrix(copy=False)
    m.fit(X, Y, w, folds=part)
    assert m.folds_cached
    orc = OracleCVMatrix(copy=False)
    orc.fit(X, Y, w)
    assert np.array_equal(m.XTX, m.XTX.T) and rel_fro(m.XTX, orc.XTX) <= 1e-12 and rel_fro(m.XTY, orc.XTY) <= 1e-11
    out = m.training_batch()
    r = orc.fold(part.get_validation_indices(2))
    assert np.array_equal(out["XTX"][2], out["XTX"][2].T)
    assert rel_fro(out["XTX"][2], r.XTX) <= 1e-12 and rel_fro(out["XTY"][2], r.XTY) <= 1e-11
    for s in STATS:
        assert np.array_equal(out[s][2], getattr(r, s)), s


@pytest.mark.parametrize("K", KS)
def test_diagonal_bands_float32_dmma(K):
    from cvmatrix_b200 import CVMatrix, Partitioner

    N, M = 6_000, 10
    X, Y, w = _inputs(N, K, M, seed=K + 303, dtype=np.float32)
    flags = (False, False, False, False)   # raw products: the regime where numpy-float32 is itself accurate
    old = os.environ.get("CVMX_F32_TC")
    os.environ["CVMX_F32_TC"] = "0"         # read when the handle is created: k_gram<float> at every K
    try:
        m = CVMatrix(*flags, dtype=np.float32)
    finally:
        if old is None:
            del os.environ["CVMX_F32_TC"]
        else:
            os.environ["CVMX_F32_TC"] = old
    m.fit(X, Y, w)
    orc = OracleCVMatrix(*flags, dtype=np.float32)
    orc.fit(X, Y, w)
    assert np.array_equal(m.XTX, m.XTX.T) and rel_fro(m.XTX, orc.XTX) <= 1e-5
    for P in (2, 60):
        folds = np.arange(N) % P
        m.set_folds(Partitioner(folds))
        out = m.training_batch()
        r = orc.fold(np.flatnonzero(folds == 1))
        XTX = out["XTX"][1]
        assert XTX.dtype == np.float32 and np.array_equal(XTX, XTX.T)
        assert rel_fro(XTX, r.XTX) <= 1e-5 and rel_fro(out["XTY"][1], r.XTY) <= 1e-5
