"""
TEST INFRASTRUCTURE - NOT PRODUCT CODE.

numpy / LAPACK restatement of the cross-validated ridge regression that ``cvmatrix_b200.CVMatrix.ridge_cross_validate``
runs on the GPU (include/cvmx.h, cvmx_ridge_cv): per penalty lam, B = (XTX + lam I)^-1 XTY on given ``XTX`` / ``XTY``
by LAPACK's Cholesky factorisation (dpotrf, lower) and solve (dpotrs), everything in float64.  ``info`` is dpotrf's:
0, or the 1-based order of the first leading minor that is not positive definite; such a penalty gets NaN
coefficients.  Prediction and PRESS are pls_oracle.predict / press, which take a stack of coefficients.
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
