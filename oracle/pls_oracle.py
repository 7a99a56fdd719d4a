"""
TEST INFRASTRUCTURE - NOT PRODUCT CODE.

numpy restatement of the cross-validated PLS that ``cvmatrix_b200.CVMatrix.pls_cross_validate`` runs on the GPU
(include/cvmx.h, cvmx_pls_cv): Improved Kernel PLS, Algorithm 2 (Dayal & MacGregor, J. Chemometrics 11:73-85, 1997)
on given ``XTX`` / ``XTY``, and the weighted PRESS of given validation rows with given training statistics.
Everything is evaluated in float64; ikpls, predict and press take a `dtype` for an extended-precision run.

    XTY_0 = XTY
    for a = 0 .. A-1:
        v = XTY_a                                     (M == 1)
        v = XTY_a q, q = dominant eigenvector of XTY_a^T XTY_a                    (M > 1)
        if ||v|| <= 64 eps ||XTY_0||_F: stop      (n_fitted = a; later B repeat the last one, B_{-1} = 0)
        w = v / ||v||;  r = w - sum_{j<a} (p_j^T w) r_j
        u = XTX r;  tTt = r^T u                       (tTt <= 0: stop as above)
        p = u / tTt;  q_a = XTY_a^T r / tTt;  XTY_{a+1} = XTY_a - tTt p q_a^T
        B_a = B_{a-1} + r q_a^T

    prediction with a + 1 components:  y^ = ((x - mu_X) / sigma_X) B_a * sigma_Y + mu_Y
"""

from __future__ import annotations

import numpy as np

EPS64 = np.finfo(np.float64).eps


def ikpls(XTX, XTY, n_components, dtype=np.float64):
    """-> (B [A, K, M], n_fitted) for one fold, evaluated in `dtype` (np.longdouble for an extended-precision run; the
    eigenvector of an M > 1 step is then float64 eigh's refined by power iterations in `dtype`)."""
    XTX = np.asarray(XTX).astype(dtype)
    XTY = np.asarray(XTY).astype(dtype).reshape(XTX.shape[0], -1)
    K, M = XTY.shape
    A = int(n_components)
    B = np.zeros((A, K, M), dtype)
    R, Pm = [], []
    Bc = np.zeros((K, M), dtype)
    y0 = np.linalg.norm(XTY)
    n_fitted = 0
    for a in range(A):
        if M == 1:
            v = XTY[:, 0].copy()
        else:
            S = XTY.T @ XTY
            _, vecs = np.linalg.eigh(S.astype(np.float64))
            q = vecs[:, -1].astype(dtype)
            if dtype != np.float64:
                for _ in range(8):
                    q = S @ q
                    q = q / np.sqrt(q @ q)
            v = XTY @ q
        nv = np.linalg.norm(v)
        if nv <= 64 * EPS64 * y0:
            break
        w = v / nv
        r = w.copy()
        for pj, rj in zip(Pm, R):
            r -= (pj @ w) * rj
        u = XTX @ r
        tTt = r @ u
        if not tTt > 0:
            break
        p = u / tTt
        q = (XTY.T @ r) / tTt
        XTY = XTY - tTt * np.outer(p, q)
        Bc = Bc + np.outer(r, q)
        R.append(r)
        Pm.append(p)
        B[a] = Bc
        n_fitted = a + 1
    B[n_fitted:] = Bc
    return B, n_fitted


def predict(Xv, B, X_mean=None, X_std=None, Y_mean=None, Y_std=None, dtype=np.float64):
    """Predictions [A, n, M] of the rows Xv with every B[a], evaluated in `dtype` (np.longdouble for an extended-precision
    reference); a statistic that is None is not applied."""
    Xt = np.asarray(Xv).astype(dtype)
    if X_mean is not None:
        Xt = Xt - np.asarray(X_mean).astype(dtype).reshape(1, -1)
    if X_std is not None:
        Xt = Xt / np.asarray(X_std).astype(dtype).reshape(1, -1)
    Yh = np.einsum("nk,akm->anm", Xt, np.asarray(B).astype(dtype))
    if Y_std is not None:
        Yh = Yh * np.asarray(Y_std).astype(dtype).reshape(1, 1, -1)
    if Y_mean is not None:
        Yh = Yh + np.asarray(Y_mean).astype(dtype).reshape(1, 1, -1)
    return Yh


def press(Xv, Yv, wv, B, X_mean=None, X_std=None, Y_mean=None, Y_std=None, dtype=np.float64):
    """Weighted PRESS [A, M] of the validation rows (wv None: unit weights), evaluated in `dtype`."""
    Yv = np.asarray(Yv).astype(dtype).reshape(np.shape(Xv)[0], np.shape(B)[2])
    wv = np.ones(Yv.shape[0], dtype) if wv is None else np.asarray(wv).astype(dtype).reshape(-1)
    res = Yv[None] - predict(Xv, B, X_mean, X_std, Y_mean, Y_std, dtype)
    return np.einsum("n,anm->am", wv, res * res)


def fold_stats(flags, X_mean, X_std, Y_mean, Y_std):
    """The statistics the prediction applies for flags = center_X | center_Y << 1 | scale_X << 2 | scale_Y << 3."""
    return (X_mean if flags & 1 else None, X_std if flags & 4 else None,
            Y_mean if flags & 2 else None, Y_std if flags & 8 else None)
