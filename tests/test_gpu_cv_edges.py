"""
GPU tests (-m gpu) of cross-validated ridge and PLS at the boundaries their kernels are built around: 64-column panels
and tiles of the ridge factorisation, one back-substitution thread per response up to M = 128, PRESS column tiles of 64
(penalty, response) columns and PRESS split over several launches, 32-row validation chunks, 64-component PRESS tiles
and 32-column K tiles of PLS, and the eigen step at M up to 128.  Ridge is compared with an extended-precision
(np.longdouble) Cholesky solve of the engine's own training matrices, so the whole tolerance measures the kernels;
PLS with the numpy IKPLS oracle.  Device outputs, windows and passes are checked bit for bit: a fold's or a penalty's
outputs do not depend on the range, the window or the pass they are computed in.
"""

import ctypes as C

import numpy as np
import pytest

import pls_oracle as po
import ridge_oracle as ro

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
C_RIDGE = 50.0       # B and PRESS of ridge to C_RIDGE kappa eps64 (kappa: 2-norm condition number of XTX + lambda I)
MAX_BOUND = 1e-8     # no compared pair may have a bound looser than this: a case never passes vacuously
WORST = []           # err / (kappa eps64) over the ridge panel sweep, printed by the sweep's last case


def _inputs(N, K, M, seed, weighted=True, dtype=np.float64):
    """Responses with a planted linear signal (decaying over the response columns) plus noise; some zero weights."""
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


def _plan(K, M, L, P, dtype=np.float64, out="numpy", want_B=False):
    """cvmx_ridge_plan of a call: folds per window W, penalties per pass Lp, PRESS chunks per launch G."""
    from cvmatrix_b200 import _lib

    plan = np.zeros(_lib.RIDGE_PLAN_LEN, np.int64)
    rc = _lib.load().cvmx_ridge_plan(K, M, L, P, _lib.F64 if dtype == np.float64 else _lib.F32,
                                     _lib.HOST if out == "numpy" else _lib.DEVICE, int(want_B), plan.ctypes.data_as(C.c_void_p))
    assert rc == _lib.OK and plan[_lib.RIDGE_FEASIBLE] == 1
    return (int(plan[_lib.RIDGE_FOLDS_PER_WINDOW]), int(plan[_lib.RIDGE_PENALTIES_PER_PASS]),
            int(plan[_lib.RIDGE_CHUNKS_PER_LAUNCH]))


def _scale(m):
    """trace(XTX) / K of the first fold: the penalty scale of the data."""
    XTX = m.training_batch(0, 1)["XTX"][0].astype(np.float64)
    return np.trace(XTX) / XTX.shape[0]


def _val(m, f):
    return m._fold_indices[m._offsets[f]:m._offsets[f + 1]]


def _ridge_ref(m, X, Y, w, alphas, f0=0, f1=None):
    """Extended-precision ridge + PRESS of folds [f0, f1) on the engine's own training matrices and statistics:
    per fold (B, info, press, sum_w_val, kappa), B and press as np.longdouble."""
    f1 = m._n_folds if f1 is None else f1
    tb = m.training_batch(f0, f1, check=False)
    out = []
    for i in range(f1 - f0):
        val = _val(m, f0 + i)
        XTX = tb["XTX"][i].astype(np.float64)
        B, info = ro.ridge_extended(XTX, tb["XTY"][i], alphas)
        g = lambda k: None if tb[k] is None else tb[k][i]  # noqa: E731
        stats = ro.fold_stats(m._flags, g("X_mean"), g("X_std"), g("Y_mean"), g("Y_std"))
        wv = None if w is None else w[val]
        ev = np.linalg.eigvalsh(XTX)
        kappa = np.array([(ev[-1] + a) / (ev[0] + a) if ev[0] + a > 0 else np.inf for a in alphas])
        pr = ro.press(X[val], Y[val], wv, np.where(np.isnan(B), 0, B), *stats, dtype=np.longdouble)
        out.append((B, info, pr, len(val) if w is None else w[val].astype(np.float64).sum(), kappa))
    return out


def _rel(a, b):
    """||a - b|| / ||b||, with b possibly np.longdouble."""
    b = np.asarray(b)
    nb = float(np.sqrt((b.astype(np.longdouble) ** 2).sum()))
    d = float(np.sqrt(((np.asarray(a).astype(np.longdouble) - b) ** 2).sum()))
    return d / (nb if nb > 0 else 1.0)


def _compare_ridge(r, ref, f0=0, cols=None, check_B=True, extra=0.0, worst=None):
    """info exactly; B and PRESS to C_RIDGE kappa eps64 (+ `extra` for outputs rounded to float32), each bound asserted
    <= MAX_BOUND.  `cols`: the penalties of r that the reference's penalties are (default: all)."""
    for i, (B, info, pr, sw, kappa) in enumerate(ref):
        f = f0 + i
        cl = np.arange(len(info)) if cols is None else np.asarray(cols)
        assert np.array_equal(r["info"][f][cl], info), (f, r["info"][f][cl], info)
        assert abs(float(r["sum_w_val"][f]) - sw) <= 1e-6 * max(sw, 1.0)
        for l, c in enumerate(cl):
            if info[l]:
                assert np.isnan(r["press"][f, c]).all()
                if check_B:
                    assert np.isnan(r["B"][f, c]).all()
                continue
            bound = C_RIDGE * kappa[l] * EPS
            assert bound <= MAX_BOUND, (f, l, kappa[l])
            e = _rel(r["press"][f, c], pr[l])
            assert e <= bound + extra, (f, l, e, bound)
            if worst is not None:
                worst.append(e / (kappa[l] * EPS))
            if check_B:
                e = _rel(r["B"][f, c], B[l])
                assert e <= bound + extra, (f, l, e, bound)
                if worst is not None:
                    worst.append(e / (kappa[l] * EPS))


def _same(a, b, keys):
    for k in keys:
        x, y = a[k], b[k]
        x = x.cpu().numpy() if hasattr(x, "cpu") else x
        y = y.cpu().numpy() if hasattr(y, "cpu") else y
        assert x.dtype == y.dtype and x.shape == y.shape, k
        assert np.array_equal(x, y, equal_nan=np.issubdtype(x.dtype, np.floating)), k


RIDGE_KEYS = ("press", "sum_w_val", "info", "status")
PLS_KEYS = ("press", "sum_w_val", "n_fitted", "status")


# ---- A. ridge panel and tile sweep --------------------------------------------------------------------------------
SWEEP = [(1, 1), (1, 128), (2, 127), (63, 1), (63, 65), (64, 64), (64, 128), (65, 1), (65, 63), (127, 2), (128, 128),
         (129, 127), (191, 65), (193, 128), (520, 7), (1100, 3)]
SWEEP_F32 = {(1, 128), (63, 65), (65, 1), (128, 128), (191, 65), (520, 7)}
SWEEP_CASES = [(K, M, np.float64) for K, M in SWEEP] + [(K, M, np.float32) for K, M in SWEEP if (K, M) in SWEEP_F32]


@pytest.mark.parametrize("K,M,dtype", SWEEP_CASES, ids=[f"K{K}-M{M}-{np.dtype(d).name}" for K, M, d in SWEEP_CASES])
def test_ridge_panel_sweep(K, M, dtype):
    P = 3
    N = max(3 * K, 60) + 30
    flags = 15 if (K + M) % 2 else 3
    X, Y, w = _inputs(N, K, M, seed=1000 + 7 * K + M, dtype=dtype)
    m = _model(X, Y, w, flags=flags, dtype=dtype, folds=np.arange(N) % P)
    L = 3 if K >= 500 else 5
    a = np.logspace(-2, 2, L) * _scale(m)
    r = m.ridge_cross_validate(a, return_coefs=True)
    assert r["press"].shape == (P, L, M) and r["B"].shape == (P, L, K, M) and r["press"].dtype == dtype
    assert not r["info"].any() and not r["status"].any()
    _compare_ridge(r, _ridge_ref(m, X, Y, w, a), extra=0.0 if dtype == np.float64 else 1e-6,
                   worst=WORST if dtype == np.float64 else None)
    if (K, M, dtype) == SWEEP_CASES[len(SWEEP) - 1]:
        print(f"\nridge panel sweep (float64): worst err / (kappa eps64) = {max(WORST):.3g} over {len(WORST)} comparisons")


# ---- B. failure in a later panel ----------------------------------------------------------------------------------
def test_ridge_failure_in_later_panels():
    # fold f's training matrix has exactly one zero column, zc[f]: the column's only non-zero entry is a validation row
    # of fold f (one product: the same bits in the totals and in the fold Gram, so T - G is exactly 0)
    K, M, N, P = 130, 3, 600, 3
    zc = [64, 100, 129]
    X, Y, w = _inputs(N, K, M, seed=130)
    folds = np.arange(N) % P
    for f, c in enumerate(zc):
        X[:, c] = 0.0
        X[3 + f, c] = 3.0         # row 3 + f is in fold f and has a non-zero weight
    assert all(folds[3 + f] == f for f in range(P)) and (w[3:6] > 0).all()
    m = _model(X, Y, w, flags=3, folds=folds)   # no scaling: the zero column stays exactly zero
    s = _scale(m)
    alphas = [0.0, 0.5 * s, 0.0, 20.0 * s]
    with pytest.warns(UserWarning, match="6 \\(fold, penalty\\) pair"):
        r = m.ridge_cross_validate(alphas, return_coefs=True)
    for f, c in enumerate(zc):
        assert list(r["info"][f]) == [c + 1, 0, c + 1, 0], (f, r["info"][f])
        assert (r["B"][f, [1, 3], c, :] == 0).all()
    _compare_ridge(r, _ridge_ref(m, X, Y, w, alphas))


# ---- C. PRESS column tiles and PRESS over several launches --------------------------------------------------------
@pytest.mark.parametrize("L,M", [(63, 1), (1, 64), (64, 1), (1, 65), (5, 13), (2, 64), (129, 1)])
def test_ridge_press_column_tiles(L, M):
    K, N, P = 40, 400, 4
    X, Y, w = _inputs(N, K, M, seed=40 + L * M)
    m = _model(X, Y, w, folds=np.arange(N) % P)
    a = np.logspace(-1.5, 1.5, L) * _scale(m)
    r = m.ridge_cross_validate(a, return_coefs=True)
    _compare_ridge(r, _ridge_ref(m, X, Y, w, a))


def test_ridge_press_over_several_launches():
    # K = 4, M = 128, L = 1024: 131,072 (penalty, response) columns leave room for 255 chunks of partials per launch, so
    # two folds of 10,000 rows (313 chunks each) take three launches and each fold straddles a launch boundary
    K, M, L, P, n = 4, 128, 1024, 2, 10_000
    W, Lp, G = _plan(K, M, L, P)
    nch = P * -(-n // 32)
    assert W == P and Lp == L and G == 255 and nch > 2 * G
    X, Y, w = _inputs(P * n, K, M, seed=404)
    m = _model(X, Y, w, folds=np.arange(P * n) % P)
    a = np.logspace(-3, 3, L) * _scale(m)
    r = m.ridge_cross_validate(a)
    sub = np.r_[0, 1, 511, 512, L - 1]
    _compare_ridge(r, _ridge_ref(m, X, Y, w, a[sub]), cols=sub, check_B=False)
    tb = m.training_batch(0, P)
    for f in range(P):
        # alone, a fold's 313 chunks take two launches split at another chunk: the same bits
        tf = m.training_batch(f, f + 1)
        assert np.array_equal(tf["XTX"][0], tb["XTX"][f]) and np.array_equal(tf["XTY"][0], tb["XTY"][f])
        rf = m.ridge_cross_validate(a, fold_begin=f, fold_end=f + 1)
        for k in RIDGE_KEYS:
            assert np.array_equal(rf[k][0], r[k][f]), (f, k)


# ---- D. validation-set sizes on the 32-row chunk edges, weighted and unweighted -----------------------------------
@pytest.mark.parametrize("weighted", [True, False], ids=["weighted", "unweighted"])
def test_validation_chunk_edges(weighted):
    sizes = [1, 31, 32, 33, 64, 65]
    K, M, N = 20, 3, 400
    X, Y, w = _inputs(N, K, M, seed=32, weighted=weighted)
    perm = np.random.default_rng(5).permutation(N)
    bounds = np.cumsum([0] + sizes)
    sets = [perm[bounds[i]:bounds[i + 1]] for i in range(len(sizes))]
    m = _model(X, Y, w, sets=sets)
    a = np.logspace(-2, 2, 4) * _scale(m)
    r = m.ridge_cross_validate(a, return_coefs=True)
    if not weighted:
        assert np.array_equal(r["sum_w_val"], np.array(sizes, np.float64))
    _compare_ridge(r, _ridge_ref(m, X, Y, w, a))
    A = 6
    rp = m.pls_cross_validate(A, return_coefs=True)
    if not weighted:
        assert np.array_equal(rp["sum_w_val"], np.array(sizes, np.float64))
    _compare_pls(rp, _pls_ref(m, X, Y, w, A), 1e-10, 1e-9)


# ---- E / F. device outputs across windows and passes; invariance over ranges, windows and passes ------------------
@pytest.fixture(scope="module")
def passes_case():
    # K = 400, L = 1024: one fold with all penalties exceeds the ~1 GiB pass, so every fold is its own window and its
    # penalties go in passes, for host and for device outputs
    K, M, L, P = 400, 2, 1024, 3
    for out in ("numpy", "torch"):
        for want_B in (False, True):
            W, Lp, _ = _plan(K, M, L, P, out=out, want_B=want_B)
            assert W == 1 and 1 < Lp < L, (out, want_B, W, Lp)
    X, Y, w = _inputs(1500, K, M, seed=31)
    m = _model(X, Y, w, folds=np.arange(1500) % P)
    a = np.logspace(-3, 3, L) * _scale(m)
    return m, (X, Y, w), a, m.ridge_cross_validate(a, return_coefs=True)


@pytest.mark.parametrize("coefs", [False, True], ids=["press", "coefs"])
def test_ridge_device_outputs_over_windows(coefs):
    # leave-one-out over 600 rows, folds 5 .. 599: four windows of ~185 folds, split differently for host and device
    # outputs; out="torch" writes each window's outputs straight into the caller's tensors at its offset
    K, M, L, N, f0 = 200, 8, 16, 600, 5
    for out in ("numpy", "torch"):
        W, Lp, _ = _plan(K, M, L, N - f0, out=out, want_B=coefs)
        assert Lp == L and 3 <= -(-(N - f0) // W) <= 5, (out, W)
    X, Y, w = _inputs(N, K, M, seed=600)
    m = _model(X, Y, w, folds=np.arange(N))
    a = np.logspace(-2, 2, L) * _scale(m)
    rh = m.ridge_cross_validate(a, fold_begin=f0, return_coefs=coefs)
    rd = m.ridge_cross_validate(a, fold_begin=f0, return_coefs=coefs, out="torch")
    _same(rh, rd, RIDGE_KEYS + (("B",) if coefs else ()))
    # folds on both sides of the first window's end (fold 183 or 189 of the range)
    _compare_ridge(rh, _ridge_ref(m, X, Y, w, a, f0 + 180, f0 + 192), f0=180, check_B=coefs)


@pytest.mark.parametrize("coefs", [False, True], ids=["press", "coefs"])
def test_ridge_device_outputs_over_passes(passes_case, coefs):
    m, _, a, r = passes_case
    rh = m.ridge_cross_validate(a, return_coefs=coefs) if not coefs else r
    rd = m.ridge_cross_validate(a, return_coefs=coefs, out="torch")
    _same(rh, rd, RIDGE_KEYS + (("B",) if coefs else ()))
    rd1 = m.ridge_cross_validate(a, fold_begin=1, return_coefs=coefs, out="torch")
    for k in RIDGE_KEYS + (("B",) if coefs else ()):
        assert np.array_equal(rd1[k].cpu().numpy(), rh[k][1:]), k


@pytest.mark.parametrize("coefs", [False, True], ids=["press", "coefs"])
def test_pls_device_outputs_over_windows(coefs):
    # leave-one-out, K = 256: about 0.6 MB of device scratch per fold, so 2500 folds take two ~1 GiB windows
    X, Y, w = _inputs(2500, 256, 2, seed=77)
    m = _model(X, Y, w, folds=np.arange(2500))
    rh = m.pls_cross_validate(4, fold_begin=3, return_coefs=coefs)
    rd = m.pls_cross_validate(4, fold_begin=3, return_coefs=coefs, out="torch")
    _same(rh, rd, PLS_KEYS + (("B",) if coefs else ()))
    if coefs:
        # a fold alone, on both sides of the first window's end (near fold 1945), and inside a short range
        for f0, f1 in ((1940, 1941), (1950, 1951), (1930, 1960)):
            rf = m.pls_cross_validate(4, fold_begin=f0, fold_end=f1, return_coefs=True)
            for k in PLS_KEYS + ("B",):
                assert np.array_equal(rf[k], rh[k][f0 - 3:f1 - 3]), (f0, k)
        _compare_pls(rh, _pls_ref(m, X, Y, w, 4, 1940, 1950), 1e-10, 1e-9, f0=1937)


def test_ridge_fold_invariance():
    # a fold alone, inside a sub-range and inside the full range of a multi-fold window: the same bits
    K, M, L, N, P = 70, 5, 6, 700, 7
    W, Lp, _ = _plan(K, M, L, P, want_B=True)
    assert W == P and Lp == L
    X, Y, w = _inputs(N, K, M, seed=70)
    m = _model(X, Y, w, folds=np.arange(N) % P)
    a = np.logspace(-2, 2, L) * _scale(m)
    r = m.ridge_cross_validate(a, return_coefs=True)
    for f0, f1 in ((0, 1), (3, 4), (6, 7), (2, 5)):
        rs = m.ridge_cross_validate(a, fold_begin=f0, fold_end=f1, return_coefs=True)
        for k in RIDGE_KEYS + ("B",):
            assert np.array_equal(rs[k], r[k][f0:f1]), (f0, f1, k)


def test_ridge_fold_and_penalty_invariance_across_passes(passes_case):
    m, (X, Y, w), a, r = passes_case
    L = len(a)
    _, Lp, _ = _plan(400, 2, L, 3, want_B=True)
    # a fold alone (its own window in both calls) and a penalty alone (every fold in one window, one penalty per pass)
    for f in range(3):
        rs = m.ridge_cross_validate(a, fold_begin=f, fold_end=f + 1, return_coefs=True)
        for k in RIDGE_KEYS + ("B",):
            assert np.array_equal(rs[k][0], r[k][f]), (f, k)
    for l in (0, Lp - 1, Lp, L - 1):
        rl = m.ridge_cross_validate(a[l:l + 1], return_coefs=True)
        for k in ("press", "info", "B"):
            assert np.array_equal(rl[k][:, 0], r[k][:, l]), (l, k)
        assert np.array_equal(rl["sum_w_val"], r["sum_w_val"])
    sub = np.r_[0, Lp - 1, Lp, L - 1]
    _compare_ridge(r, _ridge_ref(m, X, Y, w, a[sub]), cols=sub)


# ---- G. PLS edges --------------------------------------------------------------------------------------------------
def _pls_ref(m, X, Y, w, A, f0=0, f1=None):
    """IKPLS oracle + PRESS of folds [f0, f1) on the engine's own training matrices and statistics."""
    f1 = m._n_folds if f1 is None else f1
    tb = m.training_batch(f0, f1)
    X64, Y64 = X.astype(np.float64), Y.astype(np.float64)
    out = []
    for i in range(f1 - f0):
        val = _val(m, f0 + i)
        B, nf = po.ikpls(tb["XTX"][i], tb["XTY"][i], A)
        g = lambda k: None if tb[k] is None else tb[k][i].astype(np.float64)  # noqa: E731
        stats = po.fold_stats(m._flags, g("X_mean"), g("X_std"), g("Y_mean"), g("Y_std"))
        wv = None if w is None else w[val].astype(np.float64)
        out.append((B, nf, po.press(X64[val], Y64[val], wv, B, *stats), len(val) if w is None else wv.sum()))
    return out


def _compare_pls(r, ref, tol_b, tol_p, f0=0, check_B=True):
    """n_fitted exactly; press and B of component a to tol_p / tol_b, scalars or callables (fold index i, a) -> tol."""
    tb = tol_b if callable(tol_b) else lambda i, a: tol_b  # noqa: E731
    tp = tol_p if callable(tol_p) else lambda i, a: tol_p  # noqa: E731
    for i, (B, nf, pr, sw) in enumerate(ref):
        f = f0 + i
        assert r["n_fitted"][f] == nf, (f, r["n_fitted"][f], nf)
        assert abs(float(r["sum_w_val"][f]) - sw) <= 1e-6 * max(sw, 1.0)
        for a in range(B.shape[0]):
            assert _rel(r["press"][f, a], pr[a]) <= tp(i, a), (f, a, _rel(r["press"][f, a], pr[a]), tp(i, a))
            if check_B:
                assert _rel(r["B"][f, a], B[a]) <= tb(i, a), (f, a, _rel(r["B"][f, a], B[a]), tb(i, a))


def _pls_spread(m, X, Y, w, A, ref):
    """Per fold and component: the float64 oracle's own error in B and press - the larger of its distance from an
    np.longdouble run of the same algorithm and of how far it moves when XTX is perturbed by about one ulp (a
    symmetric relative perturbation of 1.1e-16 per entry, fixed seed)."""
    tb = m.training_batch()
    rng = np.random.default_rng(0)
    out = []
    for i, (B, _, pr, _) in enumerate(ref):
        XTX = tb["XTX"][i].astype(np.float64)
        E = rng.standard_normal(XTX.shape) * np.abs(XTX) * 1.1e-16
        Bp, _ = po.ikpls(XTX + (E + E.T) / 2, tb["XTY"][i], A)
        Be, _ = po.ikpls(XTX, tb["XTY"][i], A, dtype=np.longdouble)
        val = _val(m, i)
        g = lambda k: None if tb[k] is None else tb[k][i].astype(np.float64)  # noqa: E731
        stats = po.fold_stats(m._flags, g("X_mean"), g("X_std"), g("Y_mean"), g("Y_std"))
        wv = None if w is None else w[val]
        pp = po.press(X[val], Y[val], wv, Bp, *stats)
        pe = po.press(X[val], Y[val], wv, Be, *stats, dtype=np.longdouble)
        out.append(([max(_rel(Bp[a], B[a]), _rel(B[a], Be[a])) for a in range(A)],
                    [max(_rel(pp[a], pr[a]), _rel(pr[a], pe[a])) for a in range(A)]))
    return out


def _pls_case(N, K, M, A, dtype, seed, P=3, sensitive=False):
    X, Y, w = _inputs(N, K, M, seed=seed, dtype=dtype)
    m = _model(X, Y, w, dtype=dtype, folds=np.arange(N) % P)
    r = m.pls_cross_validate(A, return_coefs=True)
    assert r["press"].shape == (P, A, M) and r["B"].shape == (P, A, K, M) and r["press"].dtype == dtype
    assert not r["status"].any() and (r["n_fitted"] == A).all()
    tol = (1e-10, 1e-9) if dtype == np.float64 else (2e-5, 2e-5)
    ref = _pls_ref(m, X, Y, w, A)
    if sensitive:
        # past ~64 components of a multi-response model the dominant eigenvalues of XTY_a^T XTY_a crowd together and
        # the direction of a component becomes sensitive to rounding.  An np.longdouble run of the same algorithm on
        # these folds (M = 5, 400 training rows, K = 300) moves B by up to 8e-10 at a = 100 and 6e-8 at a = 129 from
        # the float64 oracle, and a one-ulp perturbation of XTX moves the float64 oracle by as much (up to 7e-8), while
        # at M = 1 both stay below 2e-14.  So beyond the fixed tolerance a component may differ by 10x the float64
        # oracle's own measured error at that component (_pls_spread); for the first tile of 64 components that error
        # is about 1e-12 or less and the fixed tolerance holds.
        sp = _pls_spread(m, X, Y, w, A, ref)
        tol = (lambda i, a: max(1e-10, 10 * sp[i][0][a]), lambda i, a: max(1e-9, 10 * sp[i][1][a]))
    _compare_pls(r, ref, *tol)


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["float64", "float32"])
@pytest.mark.parametrize("M", [2, 33, 64, 65, 100, 128])
def test_pls_response_counts(M, dtype):
    # the eigen step keeps S (M x M) in shared memory; k_pls_update splits rows into 256 / M groups
    _pls_case(450, 100, M, 6, dtype, seed=500 + M)


@pytest.mark.parametrize("M", [1, 5])
@pytest.mark.parametrize("A", [63, 64, 65, 129])
def test_pls_component_tiles(A, M):
    # PRESS walks the components in tiles of 64 and carries the predictions from one tile to the next; 400 training
    # rows of 300 columns keep every fold far above the early-stop threshold up to A = 129
    _pls_case(600, 300, M, A, np.float64, seed=300 + M, sensitive=M > 1)


PLS_K = [(1, 1), (31, 8), (32, 8), (33, 8), (127, 8), (128, 8), (129, 8), (1000, 5)]


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["float64", "float32"])
@pytest.mark.parametrize("K,A", PLS_K)
def test_pls_column_tiles(K, A, dtype):
    # PRESS_KT = 32-column tiles of x~ R^T and the 128-column unroll of k_pls_xtx_r
    _pls_case(max(2 * K, 120) + 30, K, 3, A, dtype, seed=900 + K)
