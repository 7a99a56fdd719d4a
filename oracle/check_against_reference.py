"""
TEST INFRASTRUCTURE.  Pins oracle/cvmatrix_oracle.py to the reference (sm00thix/cvmatrix v3.2.1).

For every combination of (center_X, center_Y, scale_X, scale_Y) x {weights with zeros, no weights} x ddof {0, 1}
x {Y, no Y} x dtype {f64, f32}, plus degenerate folds, 1-D integer input, negative weights and Partitioner
dictionaries, `grid_outputs` collects the fit attributes, training_XTX / training_XTY / training_XTX_XTY /
training_statistics of seven validation sets, and the error messages.  The live check demands *bit-identical*
outputs of the reference and the oracle in both summation orders ("numpy", "explicit").

    python oracle/check_against_reference.py                 exit code 0 = pinned (needs the reference)
    python oracle/check_against_reference.py --record PATH   stores the reference's grid outputs (.npz) for
                                                             tests/test_oracle.py, which checks them offline

The reference is looked up in $CVMATRIX_REFERENCE, else in oracle/_ref (staged by `make -C oracle ref`).
`--record PATH --from-oracle` stores the grid outputs of the oracle (order "numpy") instead and says so in the file.
"""

import itertools
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
REF = os.environ.get("CVMATRIX_REFERENCE", os.path.join(HERE, "_ref"))
STATS = ("X_mean", "X_std", "Y_mean", "Y_std")


def _put_call(out, key, f, *args):
    """Records f(*args) under key: matrices and statistics as arrays, None as '<None>', a ValueError as its message."""
    try:
        res = f(*args)
    except ValueError as e:
        out[key + "/ValueError"] = np.array(str(e))
        return
    if not isinstance(res, tuple):                                                # fit
        out[key] = np.array("<returned>")
        return
    if len(res) == 2 and isinstance(res[1], tuple):                               # (matrices, statistics)
        mats = res[0] if isinstance(res[0], tuple) else (res[0],)
        names = ("XTX", "XTY") if len(mats) == 2 else (("XTY",) if f.__name__ == "training_XTY" else ("XTX",))
        parts = list(zip(names, mats)) + list(zip(STATS, res[1]))
    else:                                                                         # training_statistics
        parts = list(zip(STATS, res))
    for name, a in parts:
        out[f"{key}/{name}"] = np.array("<None>") if a is None else np.asarray(a)


def grid_outputs(make_cv, Partitioner):
    """Every output of the pinning grid, keyed by what produced it.  make_cv(*flags, ddof=, dtype=) builds a model."""
    out = {}
    rng = np.random.default_rng(7)
    N, K, M = 403, 9, 3
    X0 = rng.normal(size=(N, K)) + 3.0
    X0[:, 4] = 2.5  # constant column -> std replaced by 1
    Y0 = rng.normal(size=(N, M)) * 10
    w0 = rng.random(N)
    w0[rng.random(N) < 0.15] = 0.0
    labels = rng.integers(0, 7, size=N)

    # Partitioner: integer labels, mixed hashables, LOO
    for i, folds in enumerate((labels, list(labels), [0, "one", 2, 2, "one", 1.0, True], np.arange(50))):
        d = Partitioner(folds).folds_dict
        out[f"part{i}/keys"] = np.array(repr(list(d.keys())))
        for j, v in enumerate(d.values()):
            out[f"part{i}/{j}"] = np.asarray(v)

    part = Partitioner(labels)
    val_sets = [part.get_validation_indices(f) for f in list(part.folds_dict)[:4]]
    val_sets.append(np.array([5]))  # single row
    val_sets.append(np.array([17, 3, 3, 250, -1]))  # unsorted, duplicate, negative
    val_sets.append(np.array([], dtype=int))  # empty
    methods = ("training_XTX", "training_statistics", "training_XTY", "training_XTX_XTY")  # raise without Y: also recorded

    for dtype in (np.float64, np.float32):
        for use_w, use_Y, ddof in itertools.product((True, False), (True, False), (0, 1)):
            for flags in itertools.product((False, True), repeat=4):
                case = f"{np.dtype(dtype).name}/w{int(use_w)}y{int(use_Y)}d{ddof}/" + "".join("TF"[not f] for f in flags)
                m = make_cv(*flags, ddof=ddof, dtype=dtype)
                m.fit(X0, Y0 if use_Y else None, w0 if use_w else None)
                for attr in ("XTX", "XTY", "sum_X", "sum_Y", "sum_sq_X", "sum_sq_Y"):
                    a = getattr(m, attr)
                    out[f"{case}/fit/{attr}"] = np.array("<None>") if a is None else np.asarray(a)
                if any(flags):
                    out[f"{case}/fit/sum_w"] = np.asarray(m.sum_w)
                    out[f"{case}/fit/sum_w_type"] = np.array(type(m.sum_w).__name__)
                    if use_w:
                        out[f"{case}/fit/nnz_w"] = np.asarray(m.num_nonzero_w)
                for j, val in enumerate(val_sets):
                    for meth in methods:
                        _put_call(out, f"{case}/val{j}/{meth}", getattr(m, meth), val)

    # degenerate folds: every training weight zero / nnz <= ddof
    wz = np.zeros(N)
    wz[labels == 0] = 1.0
    val0 = part.get_validation_indices(0)
    keep = np.setdiff1d(np.arange(N), val0)[:1]
    wz2 = wz.copy()
    wz2[keep] = 0.5  # exactly one non-zero training weight -> nnz <= ddof
    for flags in itertools.product((False, True), repeat=4):
        tag = "".join("TF"[not f] for f in flags)
        m = make_cv(*flags, ddof=1, dtype=np.float64)
        m.fit(X0, Y0, wz)
        for meth in ("training_XTX", "training_XTY", "training_XTX_XTY", "training_statistics"):
            _put_call(out, f"allzero/{tag}/{meth}", getattr(m, meth), val0)
        m.fit(X0, Y0, wz2)
        for meth in ("training_XTX", "training_XTX_XTY", "training_statistics"):
            _put_call(out, f"nnz_le_ddof/{tag}/{meth}", getattr(m, meth), val0)

    # 1-D X / Y (K = M = 1 -> pairwise column sums), integer input, negative weights
    x1 = rng.integers(0, 50, size=300)
    y1 = rng.integers(0, 9, size=300)
    w1 = rng.integers(0, 3, size=300)
    v1 = np.arange(0, 300, 3)
    for dtype in (np.float64, np.float32):
        m = make_cv(True, True, True, True, ddof=1, dtype=dtype)
        m.fit(x1, y1, w1)
        _put_call(out, f"one_dim/{np.dtype(dtype).name}/training_XTX_XTY", m.training_XTX_XTY, v1)
    _put_call(out, "negative_weights/fit", make_cv(True, True, True, True, ddof=1, dtype=np.float64).fit, X0, Y0, -w0 - 1)
    return out


def compare(got, want, matrix_tol=None):
    """Keys of `want` that `got` does not reproduce: strings and statistics bit for bit; with matrix_tol, the
    XTX / XTY matrices to that relative Frobenius error (float32: 1e-6) instead."""
    bad = sorted(set(got) ^ set(want))
    for key in sorted(set(got) & set(want)):
        a, b = got[key], want[key]
        if a.dtype.kind in "US" or b.dtype.kind in "US":
            ok = a.dtype.kind == b.dtype.kind and str(a) == str(b)
        elif a.shape != b.shape or a.dtype != b.dtype:
            ok = False
        elif matrix_tol is not None and key.rsplit("/", 1)[-1] in ("XTX", "XTY") and np.all(np.isfinite(b)):
            nb = np.linalg.norm(b.astype(np.float64))
            err = np.linalg.norm(a.astype(np.float64) - b)
            ok = err <= (matrix_tol if b.dtype == np.float64 else 1e-6) * nb
        else:
            ok = np.array_equal(a, b, equal_nan=True)
        if not ok:
            bad.append(key)
    return bad


def oracle_classes(order):
    from cvmatrix_oracle import OracleCVMatrix, OraclePartitioner

    class OracleWithRefNames(OracleCVMatrix):
        """The oracle under the reference's attribute names."""

        def __init__(self, *flags, ddof, dtype):
            super().__init__(*flags, ddof=ddof, dtype=dtype, order=order)

        @property
        def num_nonzero_w(self):
            return self.nnz_w

    return OracleWithRefNames, OraclePartitioner


def load_reference():
    if not os.path.isfile(os.path.join(REF, "cvmatrix", "cvmatrix.py")):
        return None
    sys.path.insert(0, REF)
    from cvmatrix import CVMatrix, Partitioner  # the unmodified reference

    return (lambda *flags, ddof, dtype: CVMatrix(*flags, ddof=ddof, dtype=dtype)), Partitioner


def record(path, from_oracle):
    if from_oracle:
        src = ("oracle/cvmatrix_oracle.py, order 'numpy' (found bit-identical to the reference over this grid by "
               "the live check)")
        out = grid_outputs(*oracle_classes("numpy"))
    else:
        ref = load_reference()
        if ref is None:
            print(f"reference not present at {REF}; nothing to record")
            return 2
        src = "sm00thix/cvmatrix v3.2.1 (unmodified)"
        out = grid_outputs(*ref)
    # one copy of every distinct array: many grid cells repeat one another's statistics and matrices
    index, blobs, seen = {}, [], {}
    for key, a in out.items():
        tag = (a.dtype.str, a.shape, a.tobytes())
        if tag not in seen:
            seen[tag] = len(blobs)
            blobs.append(a)
        index[key] = seen[tag]
    meta = dict(source=src, numpy=np.__version__, keys=list(index), blob_of=[index[k] for k in index])
    np.savez_compressed(path, __meta__=np.array(json.dumps(meta)), **{f"b{i}": a for i, a in enumerate(blobs)})
    print(f"{len(out)} outputs ({len(blobs)} distinct) from {src} -> {path} ({os.path.getsize(path) / 1e3:.0f} kB)")
    return 0


def load_recorded(path):
    """-> (outputs dict, source) of a file written by --record."""
    with np.load(path) as z:
        meta = json.loads(str(z["__meta__"]))
        blobs = {int(k[1:]): z[k] for k in z.files if k != "__meta__"}
    return {k: blobs[i] for k, i in zip(meta["keys"], meta["blob_of"])}, meta["source"]


def main():
    if "--record" in sys.argv:
        return record(sys.argv[sys.argv.index("--record") + 1], "--from-oracle" in sys.argv)
    ref = load_reference()
    if ref is None:
        print(f"reference not present at {REF}; nothing to pin against")
        return 2
    want = grid_outputs(*ref)
    fails = 0
    for order in ("numpy", "explicit"):
        bad = compare(grid_outputs(*oracle_classes(order)), want)
        fails += len(bad)
        for key in bad[:20]:
            print("mismatch", order, key)
    print(f"{2 * len(want)} checks, {fails} failures")
    return 0 if fails == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
