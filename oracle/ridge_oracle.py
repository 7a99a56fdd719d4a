"""
TEST INFRASTRUCTURE - NOT PRODUCT CODE.

numpy / LAPACK restatement of the cross-validated ridge regression that ``cvmatrix_b200.CVMatrix.ridge_cross_validate``
runs on the GPU (include/cvmx.h, cvmx_ridge_cv): per penalty lam, B = (XTX + lam I)^-1 XTY on given ``XTX`` / ``XTY``
by LAPACK's Cholesky factorisation (dpotrf, lower) and solve (dpotrs), everything in float64.  ``info`` is dpotrf's:
0, or the 1-based order of the first leading minor that is not positive definite; such a penalty gets NaN
coefficients.  Prediction and PRESS are pls_oracle.predict / press, which take a stack of coefficients.

``ridge_extended`` is the same solve in extended precision (``np.longdouble``, 64-bit significand on x86-64): a plain
column-by-column Cholesky factorisation with forward and back substitution, so that a comparison with the float64
kernels measures the kernels' rounding and not the reference's.
"""

from __future__ import annotations

import numpy as np
from scipy.linalg import lapack

from pls_oracle import fold_stats, predict, press  # noqa: F401  (re-exported for the tests)


def ridge(XTX, XTY, alphas):
    """-> (B [L, K, M] float64, NaN where info != 0; info [L] int32) for one fold."""
    XTX = np.asarray(XTX, np.float64)
    K = XTX.shape[0]
    XTY = np.asarray(XTY, np.float64).reshape(K, -1)
    alphas = np.asarray(alphas, np.float64).reshape(-1)
    B = np.full((alphas.size, K, XTY.shape[1]), np.nan)
    info = np.zeros(alphas.size, np.int32)
    for l, lam in enumerate(alphas):
        c, inf = lapack.dpotrf(XTX + lam * np.eye(K), lower=1, clean=1)
        info[l] = inf
        if inf == 0:
            b, inf2 = lapack.dpotrs(c, XTY, lower=1)
            assert inf2 == 0
            B[l] = b
    return B, info


def ridge_extended(XTX, XTY, alphas):
    """-> (B [L, K, M] np.longdouble, NaN where info != 0; info [L] int32) for one fold, with ``ridge``'s contract:
    info is the 1-based column of the first pivot that is not > 0."""
    ld = np.longdouble
    XTX = np.asarray(XTX).astype(ld)
    K = XTX.shape[0]
    XTY = np.asarray(XTY).astype(ld).reshape(K, -1)
    alphas = np.asarray(alphas, np.float64).reshape(-1)
    B = np.full((alphas.size, K, XTY.shape[1]), np.nan, dtype=ld)
    info = np.zeros(alphas.size, np.int32)
    for l, lam in enumerate(alphas):
        A = XTX + ld(lam) * np.eye(K, dtype=ld)
        Lc = np.zeros((K, K), dtype=ld)
        for j in range(K):
            d = A[j, j] - Lc[j, :j] @ Lc[j, :j]
            if not d > 0:
                info[l] = j + 1
                break
            Lc[j, j] = np.sqrt(d)
            Lc[j + 1:, j] = (A[j + 1:, j] - Lc[j + 1:, :j] @ Lc[j, :j]) / Lc[j, j]
        if info[l]:
            continue
        z = np.zeros_like(XTY)
        for j in range(K):   # L z = XTY
            z[j] = (XTY[j] - Lc[j, :j] @ z[:j]) / Lc[j, j]
        b = np.zeros_like(XTY)
        for j in range(K - 1, -1, -1):   # L^T b = z
            b[j] = (z[j] - Lc[j + 1:, j] @ b[j + 1:]) / Lc[j, j]
        B[l] = b
    return B, info
