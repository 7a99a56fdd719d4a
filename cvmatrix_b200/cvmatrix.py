"""
CVMatrix on B200: drop-in for ``cvmatrix.CVMatrix`` (reference cvmatrix/cvmatrix.py:99-1243,
Algorithms 2-7 of Engstrøm & Jensen 2025) whose arithmetic runs in hand-written sm_100a
kernels behind the C ABI of libcvmx.so (include/cvmx.h).  There is no CPU fallback: the
class raises at construction when the CUDA library or a B200 is missing.

Same constructor options (center_X, center_Y, scale_X, scale_Y, ddof, dtype, copy), same
methods (fit, training_XTX, training_XTY, training_XTX_XTY, training_statistics), same return
structure (fresh numpy arrays of the requested dtype; statistics as (1, K) / (1, M) rows or
None), same ValueError messages.  Beyond the reference: ``set_folds`` / ``training_batch``
evaluate many folds in one launch with device-resident outputs (the shape of the reference's
``jax.vmap`` use, benchmarks/benchmark.py:136-152).

Host code here only marshals arrays, decides which statistics a method returns
(cvmatrix/cvmatrix.py:563-574, 806-833) and turns per-fold status bits into the reference's
exceptions (cvmatrix/cvmatrix.py:625-629, 1074-1078).
"""

from __future__ import annotations

import contextlib
import ctypes as C
import warnings
from typing import Optional, Sequence, Tuple, Union

import numpy as np
from numpy import typing as npt

from . import _lib
from .partitioner import Partitioner

Array = np.ndarray
Stats = Tuple[Optional[Array], Optional[Array], Optional[Array], Optional[Array]]

_ERR_NO_NONZERO = "The number of non-zero weights in the training set must be greater than zero."
_ERR_DDOF = "The number of non-zero weights in the training set must be greater than `ddof`."
_ERR_NOTHING = "At least one of `return_XTX` and `return_XTY` must be True."
_ERR_NO_Y = "Response variables `Y` are not provided."


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _tptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class CVMatrix:
    r"""
    Parameters
    ----------
    center_X, center_Y, scale_X, scale_Y : bool, default True
        Training-set centering / scaling of X and Y inside :math:`X^T W X` and :math:`X^T W Y`
        (means and standard deviations are those of each fold's training set).
    ddof : int, default 1
        Delta degrees of freedom of the weighted standard deviation.
    dtype : np.float64 (default) or np.float32
        Model dtype.  Other floating types of the reference's numpy backend (float16, longdouble)
        have no B200 path and are rejected.
    copy : bool, default True
        Same meaning as in the reference for the host-side ``X`` / ``Y`` / ``weights`` attributes;
        the device always holds its own copy.
    backend : str, default "numpy"
        Accepted for signature compatibility.  "numpy" selects the numpy-backend *semantics*, which is
        the only thing this engine implements; "cuda" is an alias.  "jax" is rejected (no multi-backend
        dispatch here).
    device : int, optional
        CUDA device ordinal (default: the current torch device if torch is imported, else 0).
    """

    def __init__(
        self,
        center_X: bool = True,
        center_Y: bool = True,
        scale_X: bool = True,
        scale_Y: bool = True,
        ddof: int = 1,
        dtype: npt.DTypeLike = np.float64,
        copy: bool = True,
        backend: str = "numpy",
        device: Optional[int] = None,
    ) -> None:
        if backend == "jax":
            # same exception type and install hint as the reference without JAX (cvmatrix/cvmatrix.py:85-90): the JAX
            # path is the reference package's optional extra; this engine has no multi-backend dispatch
            raise ImportError("backend='jax' is the reference package's optional JAX path (`pip install cvmatrix[jax]`); "
                              "cvmatrix_b200 implements the numpy-backend semantics on B200 only.")
        if backend not in ("numpy", "cuda"):
            raise ValueError(f"Invalid backend: {backend!r}. This engine implements the numpy-backend semantics on B200 only.")
        self.center_X = center_X
        self.center_Y = center_Y
        self.scale_X = scale_X
        self.scale_Y = scale_Y
        self.ddof = ddof
        self.dtype = dtype.type if isinstance(dtype, np.dtype) else dtype
        if np.dtype(self.dtype) not in (np.dtype(np.float64), np.dtype(np.float32)):
            raise TypeError(f"dtype {np.dtype(self.dtype).name} has no B200 path; use float64 or float32")
        self.copy = copy
        self.backend = backend
        self.resolution = np.finfo(dtype).resolution * 10
        self.X = self.Y = self.weights = None
        self.N = self.K = self.M = None
        self.XTX = self.XTY = None
        self.sum_X = self.sum_Y = self.sum_sq_X = self.sum_sq_Y = None
        self.sum_w = self.num_nonzero_w = None

        self._lib = _lib.load()
        if device is None:
            device = 0
            try:
                import sys

                if "torch" in sys.modules:
                    import torch

                    if torch.cuda.is_available():
                        device = torch.cuda.current_device()
            except Exception:  # pragma: no cover
                device = 0
        self.device = int(device)
        self._flags = int(bool(center_X)) | int(bool(center_Y)) << 1 | int(bool(scale_X)) << 2 | int(bool(scale_Y)) << 3
        self._h = C.c_void_p()
        rc = self._lib.cvmx_create(
            self.device, _lib.F64 if np.dtype(self.dtype) == np.float64 else _lib.F32, self._flags, int(ddof),
            float(self.resolution), C.byref(self._h),
        )
        _lib.check(rc, None)
        self._partitioner: Optional[Partitioner] = None

    # ---- pickling (the reference object is a plain picklable container that callers ship to worker processes,
    # cvmatrix/partitioner.py:26-31): device state is dropped and rebuilt from the host arrays on load -----------
    def __getstate__(self):
        if getattr(self, "_streamed", False) and self.X is None:
            raise TypeError("a CVMatrix fitted through fit_begin / fit_rows / fit_end keeps its rows on the device only and "
                            "cannot be pickled; fit from host arrays instead")
        state = {k: v for k, v in self.__dict__.items() if k not in ("_lib", "_h", "_partitioner", "_pinned_pool")}
        if getattr(self, "_n_folds", 0) and getattr(self, "_fold_indices", None) is None:
            state["_n_folds"] = 0       # the CSR lives on the device only (should not happen: set_folds keeps a host copy)
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self._lib = _lib.load()
        self._partitioner = None
        self._h = C.c_void_p()
        rc = self._lib.cvmx_create(
            self.device, _lib.F64 if np.dtype(self.dtype) == np.float64 else _lib.F32, self._flags, int(self.ddof),
            float(self.resolution), C.byref(self._h),
        )
        _lib.check(rc, None)
        self._streamed = False
        n_folds, offsets, indices = state.get("_n_folds", 0), state.get("_offsets"), state.get("_fold_indices")
        if self.X is not None:
            keep, self.copy = self.copy, False   # the unpickled arrays are already private copies
            try:
                self.fit(self.X, self.Y, None if self.weights is None else self.weights)   # resets the fold state
            finally:
                self.copy = keep
            if n_folds and offsets is not None and indices is not None:
                self._upload_csr(offsets, indices)   # the validation sets travel with the object

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._lib.cvmx_destroy(h)
            except Exception:  # pragma: no cover - interpreter shutdown
                pass
            self._h = C.c_void_p()

    # ---- fit ---------------------------------------------------------------------------------------
    def _init_mat(self, mat) -> Array:
        # cvmatrix/cvmatrix.py:1131-1151
        mat = np.asarray(mat, dtype=self.dtype)
        if self.copy and mat.dtype == self.dtype:
            mat = mat.copy()
        if mat.ndim == 1:
            mat = mat.reshape(-1, 1)
        return mat

    @staticmethod
    def _rows(a: Array):
        """(array the library can read, leading dimension in elements): rows must be contiguous."""
        item = a.dtype.itemsize
        if (a.shape[0] > 1 and a.shape[1] > 0 and a.strides[1] == item and a.strides[0] % item == 0
                and a.strides[0] >= a.shape[1] * item):
            return a, a.strides[0] // item
        a = np.ascontiguousarray(a)
        return a, max(a.shape[1], 1)

    def fit(self, X: npt.ArrayLike, Y: Optional[npt.ArrayLike] = None, weights: Optional[npt.ArrayLike] = None,
            _gram_rows: Optional[Tuple[int, int]] = None, folds: Optional[Partitioner] = None) -> None:
        """cvmatrix/cvmatrix.py:207-328.  Uploads X, Y, weights and computes the dataset-wide totals on the GPU.

        ``folds`` (extension): a ``Partitioner`` whose validation sets are uploaded in the same call
        (= ``fit`` + ``set_folds``).  Its folds partition the rows, so every row is contracted once, per fold, behind
        the upload, and ``training_batch`` afterwards only runs the statistics and the epilogue (cvmx_fit_folds)."""
        self._streamed = False
        self.X = self._init_mat(X)
        self.N, self.K = self.X.shape
        if Y is not None:
            self.Y = self._init_mat(Y)
            self.M = self.Y.shape[1]
        else:
            self.Y = None
            self.M = None
        self.weights = self._init_mat(weights) if weights is not None else None
        if self.Y is not None and self.Y.shape[0] != self.N:
            raise ValueError("X and Y must have the same number of rows")
        if self.weights is not None and self.weights.shape[0] != self.N:
            raise ValueError("weights must have one entry per row of X")
        self._partitioner = None
        self._n_folds = 0
        self._offsets = self._fold_indices = None

        Xd, ldx = self._rows(self.X)
        Yd, ldy = self._rows(self.Y) if self.Y is not None else (None, 0)
        wd = np.ascontiguousarray(self.weights.reshape(-1)) if self.weights is not None else None
        g0, g1 = (0, self.N) if _gram_rows is None else _gram_rows
        if folds is not None:
            if _gram_rows is not None:
                raise ValueError("folds= cannot be combined with a row-sharded Gram pass")
            offsets, indices = folds.csr()
            if indices.size != self.N:
                raise ValueError("the Partitioner was built for a different number of rows")
            rc = self._lib.cvmx_fit_folds(self._h, _ptr(Xd), self.N, self.K, ldx, _ptr(Yd), self.M or 0, ldy, _ptr(wd), _lib.HOST,
                                          _ptr(offsets), _ptr(indices), offsets.size - 1, 1)
            _lib.check(rc, self._h)
            self._partitioner = folds
            self._n_folds = offsets.size - 1
            self._offsets = offsets
            self._fold_indices = indices
        else:
            rc = self._lib.cvmx_fit(self._h, _ptr(Xd), self.N, self.K, ldx, _ptr(Yd), self.M or 0, ldy, _ptr(wd), _lib.HOST, g0, g1)
            _lib.check(rc, self._h)
        self._pull_totals()

    # ---- streaming / sharded fit (include/cvmx.h: cvmx_fit_begin / cvmx_fit_rows / cvmx_fit_end) -------------------
    def fit_begin(self, N: int, K: int, M: int = 0, weighted: bool = False, max_block_rows: int = 65536) -> None:
        """Starts a fit that is fed in row blocks (``fit_rows``) and completed by ``fit_end``: for matrices that are
        produced on the device, that exceed host memory, or whose upload is shared by several GPUs."""
        self.X = self.Y = self.weights = None
        self.N, self.K, self.M = int(N), int(K), (int(M) if M else None)
        self._partitioner = None
        self._n_folds = 0
        self._offsets = self._fold_indices = None
        self._streamed = False
        self._stream_weighted = bool(weighted)
        _lib.check(self._lib.cvmx_fit_begin(self._h, int(N), int(K), int(M or 0), int(bool(weighted)), int(max_block_rows)), self._h)

    @staticmethod
    def _block(a, dtype):
        """(pointer, leading dimension, memory kind, keep-alive) of a row block: numpy array or CUDA torch tensor."""
        if a is None:
            return None, 0, None, None
        if hasattr(a, "data_ptr"):   # torch tensor
            if a.dim() == 1:
                a = a.reshape(-1, 1)
            if a.stride(-1) != 1 or (a.dim() == 2 and a.shape[0] > 1 and a.stride(0) < a.shape[1]):
                a = a.contiguous()
            if str(a.dtype).split(".")[-1] != np.dtype(dtype).name:
                raise TypeError(f"block dtype {a.dtype} does not match the model dtype {np.dtype(dtype).name}")
            ldim = a.stride(0) if (a.dim() == 2 and a.shape[0] > 1) else max(a.shape[-1], 1)
            return C.c_void_p(a.data_ptr()), int(ldim), (_lib.DEVICE if a.is_cuda else _lib.HOST), a
        a = np.asarray(a, dtype=dtype)
        if a.ndim == 1:
            a = a.reshape(-1, 1)
        a, ldim = CVMatrix._rows(a)
        return _ptr(a), int(ldim), _lib.HOST, a

    def fit_rows(self, row0: int, X, Y=None, weights=None, gram: bool = True) -> None:
        """Rows ``[row0, row0 + len(X))`` of the data set: numpy arrays (host) or CUDA torch tensors (device).  With
        ``gram`` the block's weighted Gram is added to the totals (every row by exactly one rank)."""
        xp, ldx, mem, kx = self._block(X, self.dtype)
        yp, ldy, memy, ky = self._block(Y, self.dtype)
        if weights is not None:   # the library reads nrows CONTIGUOUS weights: flatten strided views first
            weights = (weights.reshape(-1).contiguous() if hasattr(weights, "data_ptr")
                       else np.ascontiguousarray(np.asarray(weights, dtype=self.dtype).reshape(-1)))
        wp, ldw, memw, kw = self._block(weights, self.dtype)
        if wp is not None and (ldw != 1 or int(kw.shape[0]) != int(kx.shape[0])):
            raise ValueError("weights must hold one contiguous value per row of the block")
        if (yp is not None and memy != mem) or (wp is not None and memw != mem):
            raise ValueError("X, Y and weights of a block must live in the same memory (all host or all device)")
        nrows = int(kx.shape[0])
        _lib.check(self._lib.cvmx_fit_rows(self._h, int(row0), nrows, xp, ldx, yp, ldy, wp, mem, int(bool(gram))), self._h)

    def fit_end(self, col_shard: int = 0, n_col_shards: int = 1, pull: bool = True) -> None:
        """Completes a streamed fit.  Multi-GPU callers pass their column shard, all-reduce the totals and moment rows
        (``distributed.fit_sharded_upload``) and call ``_pull_totals`` themselves."""
        _lib.check(self._lib.cvmx_fit_end(self._h, int(col_shard), int(n_col_shards)), self._h)
        self._streamed = True
        if pull:
            self._pull_totals()

    def _pull_totals(self) -> None:
        dt, K, M = self.dtype, self.K, self.M or 0
        XTX = np.empty((K, K), dt)
        XTY = np.empty((K, M), dt) if M else None
        sX, qX = np.empty((1, K), dt), np.empty((1, K), dt)
        sY, qY = (np.empty((1, M), dt), np.empty((1, M), dt)) if M else (None, None)
        sum_w, nnz = C.c_double(), C.c_int64()
        rc = self._lib.cvmx_get_totals(self._h, _ptr(XTX), _ptr(XTY), _ptr(sX), _ptr(sY), _ptr(qX), _ptr(qY),
                                       C.byref(sum_w), C.byref(nnz))
        _lib.check(rc, self._h)
        cX, cY, sXf, sYf = self.center_X, self.center_Y, self.scale_X, self.scale_Y
        self.XTX, self.XTY = XTX, XTY
        # gating of the public attributes: cvmatrix/cvmatrix.py:1223-1243
        if cX or cY or sXf or sYf:
            if self._is_weighted:
                self.sum_w, self.num_nonzero_w = self.dtype(sum_w.value), int(nnz.value)
            else:
                self.sum_w, self.num_nonzero_w = self.N, self.N
        else:
            self.sum_w = self.num_nonzero_w = None
        self.sum_X = sX if (cX or cY or sXf) else None
        self.sum_Y = sY if (M and (cX or cY or sYf)) else None
        self.sum_sq_X = qX if sXf else None
        self.sum_sq_Y = qY if (M and sYf) else None

    # Derived N x K host arrays of the reference (cvmatrix/cvmatrix.py:1193-1207, 1235, 1240).  The device
    # never materialises them (products are formed in registers); they are computed on access.
    @property
    def WX(self):
        if self.X is None:
            return None
        return self.X if self.weights is None else self.X * self.weights

    @property
    def WY(self):
        if self.Y is None:
            return None
        if self.weights is None:
            return self.Y
        return self.Y * self.weights if (self.center_X or self.center_Y or self.scale_Y) else None

    @property
    def sq_X(self):
        return self.WX * self.X if (self.X is not None and self.scale_X) else None

    @property
    def sq_Y(self):
        return self.WY * self.Y if (self.Y is not None and self.scale_Y) else None

    # ---- per-call API (reference signatures) ---------------------------------------------------------
    def training_XTX(self, validation_indices: npt.NDArray[np.int_]) -> Tuple[Array, Stats]:
        """cvmatrix/cvmatrix.py:330-383"""
        return self._training_matrices(True, False, validation_indices)

    def training_XTY(self, validation_indices: npt.NDArray[np.int_]) -> Tuple[Array, Stats]:
        """cvmatrix/cvmatrix.py:385-449"""
        return self._training_matrices(False, True, validation_indices)

    def training_XTX_XTY(self, validation_indices: npt.NDArray[np.int_]) -> Tuple[Tuple[Array, Array], Stats]:
        """cvmatrix/cvmatrix.py:451-517"""
        return self._training_matrices(True, True, validation_indices)

    def training_statistics(self, validation_indices: npt.NDArray[np.int_]) -> Stats:
        """cvmatrix/cvmatrix.py:519-574"""
        self._require_fit()
        has_Y = self._has_Y
        need = (self.center_X or self.scale_X, self.scale_X, (self.center_Y or self.scale_Y) and has_Y, self.scale_Y and has_Y)
        _, _, stats = self._run_indices(validation_indices, _lib.WANT_STATS, need)
        return stats

    def _training_matrices(self, return_XTX: bool, return_XTY: bool, val_indices):
        """cvmatrix/cvmatrix.py:754-896"""
        if not return_XTX and not return_XTY:
            raise ValueError(_ERR_NOTHING)
        self._require_fit()
        if return_XTY and not self._has_Y:
            raise ValueError(_ERR_NO_Y)
        cX, cY, sX, sY = self.center_X, self.center_Y, self.scale_X, self.scale_Y
        need = (cX or (return_XTY and cY), sX, return_XTY and (cX or cY), return_XTY and sY)
        want = (_lib.WANT_XTX if return_XTX else 0) | (_lib.WANT_XTY if return_XTY else 0) | _lib.WANT_STATS
        XTX, XTY, stats = self._run_indices(val_indices, want, need)
        if return_XTX and return_XTY:
            return (XTX, XTY), stats
        return (XTX if return_XTX else XTY), stats

    @property
    def _has_Y(self) -> bool:
        return self.Y is not None or (getattr(self, "_streamed", False) and bool(self.M))

    @property
    def _is_weighted(self) -> bool:
        return self.weights is not None or (getattr(self, "_streamed", False) and getattr(self, "_stream_weighted", False))

    def _require_fit(self):
        if self.X is None and not getattr(self, "_streamed", False):
            raise ValueError("fit must be called before the training matrices can be computed")

    @staticmethod
    def _as_index_array(val) -> np.ndarray:
        val = np.asarray(val)
        if val.dtype.kind not in "iu":
            raise IndexError("arrays used as indices must be of integer type")
        if val.ndim != 1:
            val = val.reshape(-1)
        return np.ascontiguousarray(val, dtype=np.int64)

    def _raise_for_status(self, status: int, need) -> None:
        any_stat = any(need)
        if any_stat and self._is_weighted and (status & _lib.FOLD_NO_NONZERO_W):
            raise ValueError(_ERR_NO_NONZERO)
        if (need[1] or need[3]) and (status & _lib.FOLD_NNZ_LE_DDOF):
            raise ValueError(_ERR_DDOF)

    def _split_stats(self, row_pair: np.ndarray, need) -> Stats:
        K, M = self.K, self.M or 0
        mean, std = row_pair[0], row_pair[1]
        return (
            mean[:K].reshape(1, K).copy() if need[0] else None,
            std[:K].reshape(1, K).copy() if need[1] else None,
            mean[K:K + M].reshape(1, M).copy() if need[2] else None,
            std[K:K + M].reshape(1, M).copy() if need[3] else None,
        )

    def _run_indices(self, val_indices, want: int, need):
        val = self._as_index_array(val_indices)
        dt, K, M = self.dtype, self.K, self.M or 0
        XTX = np.empty((K, K), dt) if want & _lib.WANT_XTX else None
        XTY = np.empty((K, M), dt) if want & _lib.WANT_XTY else None
        stats = np.empty((2, K + M), dt)
        status = np.zeros(1, np.int32)
        rc = self._lib.cvmx_training_indices(self._h, _ptr(val), val.size, _lib.HOST, want & 3, _ptr(XTX), _ptr(XTY), _ptr(stats),
                                             None, _ptr(status), _lib.HOST)
        _lib.check(rc, self._h)
        self._raise_for_status(int(status[0]), need)
        return XTX, XTY, self._split_stats(stats, need)

    # ---- batched API -----------------------------------------------------------------------------------
    def set_folds(self, folds: Union[Partitioner, Sequence[npt.NDArray[np.int_]]]) -> None:
        """Uploads all validation index sets as one device-resident CSR (a ``Partitioner`` or a sequence
        of index arrays)."""
        self._require_fit()
        if isinstance(folds, Partitioner):
            offsets, indices = folds.csr()
        else:
            sets = [self._as_index_array(v) for v in folds]
            offsets = np.zeros(len(sets) + 1, np.int64)
            if sets:
                np.cumsum([s.size for s in sets], out=offsets[1:])
            indices = np.concatenate(sets) if sets else np.zeros(0, np.int64)
        self._upload_csr(offsets, indices)

    def _upload_csr(self, offsets, indices) -> None:
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        indices = np.ascontiguousarray(indices, dtype=np.int64)
        rc = self._lib.cvmx_set_folds(self._h, _ptr(offsets), _ptr(indices), offsets.size - 1, _lib.HOST)
        _lib.check(rc, self._h)
        self._n_folds = offsets.size - 1
        self._offsets = offsets
        self._fold_indices = indices    # host copy: pickling re-uploads it (cvmatrix/partitioner.py:26-31 ships folds separately)

    def training_batch(self, fold_begin: int = 0, fold_end: Optional[int] = None, return_XTX: bool = True,
                       return_XTY: bool = True, out: str = "numpy", check: bool = True):
        """
        All folds ``[fold_begin, fold_end)`` of the CSR in one batched launch.

        Returns a dict with ``XTX`` (P, K, K), ``XTY`` (P, K, M), ``X_mean``/``X_std`` (P, 1, K),
        ``Y_mean``/``Y_std`` (P, 1, M) (entries the flags do not define are None, exactly as the per-call
        methods decide), ``sum_w_train`` / ``nnz_train`` (P,) and ``status`` (P,) int32.
        ``out="numpy"`` copies results to fresh host arrays; ``out="pinned"`` to page-locked host arrays from a pool
        that the next ``out="pinned"`` call overwrites (10x faster for large batches); ``out="torch"`` leaves them on
        the device as torch tensors (no host copy; the consumer's next step runs on the GPU).  With ``check`` the degenerate
        fold errors of the reference are raised for the first offending fold.
        """
        self._require_fit()
        if fold_end is None:
            fold_end = self._n_folds
        if not return_XTX and not return_XTY:
            raise ValueError(_ERR_NOTHING)
        if return_XTY and not self._has_Y:
            raise ValueError(_ERR_NO_Y)
        P = fold_end - fold_begin
        dt, K, M = self.dtype, self.K, self.M or 0
        want = (_lib.WANT_XTX if return_XTX else 0) | (_lib.WANT_XTY if return_XTY else 0)
        cX, cY, sX, sY = self.center_X, self.center_Y, self.scale_X, self.scale_Y
        need = (cX or (return_XTY and cY), sX, return_XTY and (cX or cY), return_XTY and sY)
        if out == "torch":
            import torch

            tdt = torch.float64 if np.dtype(dt) == np.float64 else torch.float32
            dev = torch.device("cuda", self.device)
            XTX = torch.empty((P, K, K), dtype=tdt, device=dev) if return_XTX else None
            XTY = torch.empty((P, K, M), dtype=tdt, device=dev) if return_XTY else None
            stats = torch.empty((P, 2, K + M), dtype=tdt, device=dev)
            scal = torch.empty((P, 2), dtype=tdt, device=dev)
            status = torch.empty((P,), dtype=torch.int32, device=dev)
            p = _tptr
            mem = _lib.DEVICE
        elif out == "pinned":
            # page-locked host arrays from a pool that is REUSED by the next out="pinned" call: the device->host copy
            # then runs at the PCIe rate (a copy into fresh pageable numpy memory is bounded by page faults and the
            # driver's bounce buffer, ~5 GB/s measured)
            XTX = self._pinned("XTX", (P, K, K)) if return_XTX else None
            XTY = self._pinned("XTY", (P, K, M)) if return_XTY else None
            stats = self._pinned("stats", (P, 2, K + M))
            scal = self._pinned("scal", (P, 2))
            status = self._pinned("status", (P,), np.int32)
            p = _ptr
            mem = _lib.HOST
        elif out == "numpy":
            XTX = np.empty((P, K, K), dt) if return_XTX else None
            XTY = np.empty((P, K, M), dt) if return_XTY else None
            stats = np.empty((P, 2, K + M), dt)
            scal = np.empty((P, 2), dt)
            status = np.zeros((P,), np.int32)
            p = _ptr
            mem = _lib.HOST
        else:
            raise ValueError("out must be 'numpy', 'pinned' or 'torch'")
        with self._torch_stream() if out == "torch" else contextlib.nullcontext():
            rc = self._lib.cvmx_training_batch(self._h, fold_begin, fold_end, want, p(XTX), p(XTY), p(stats), p(scal), p(status), mem)
            _lib.check(rc, self._h)
        if check:
            st = status.cpu().numpy() if out == "torch" else status
            for s in np.unique(st):
                if s:
                    self._raise_for_status(int(s), need)
        mean, std = stats[:, 0:1, :], stats[:, 1:2, :]
        return dict(
            XTX=XTX, XTY=XTY,
            X_mean=mean[:, :, :K] if need[0] else None, X_std=std[:, :, :K] if need[1] else None,
            Y_mean=mean[:, :, K:] if need[2] else None, Y_std=std[:, :, K:] if need[3] else None,
            sum_w_train=scal[:, 0], nnz_train=scal[:, 1], status=status,
        )

    @contextlib.contextmanager
    def _torch_stream(self):
        """Runs the enclosed library calls stream-ordered with torch's current stream, so that freshly allocated torch
        outputs are safe to write.  The legacy default stream has no handle to share: the library then orders against it
        with a full synchronisation instead."""
        import torch

        ts = torch.cuda.current_stream(torch.device("cuda", self.device))
        bound = False
        if ts.cuda_stream:
            _lib.check(self._lib.cvmx_set_stream(self._h, C.c_void_p(ts.cuda_stream)), self._h)
            bound = True
        else:
            ts.synchronize()
        try:
            yield
        finally:
            if bound:   # always unbind: a failed call must not leave the handle on the caller's stream
                self._lib.cvmx_set_stream(self._h, None)  # syncs, back to the private stream
            else:       # legacy default stream: the results must be complete before torch touches them
                self._lib.cvmx_sync(self._h)

    def pls_cross_validate(self, n_components: int, fold_begin: int = 0, fold_end: Optional[int] = None,
                           return_coefs: bool = False, out: str = "numpy", check: bool = True,
                           return_predictions: bool = False):
        """
        Cross-validated PLS regression over folds ``[fold_begin, fold_end)`` of the CSR (see ``set_folds``), on the GPU.

        Every fold's model is fitted by Improved Kernel PLS (Algorithm 2 of Dayal & MacGregor, 1997) in float64 from
        the fold's ``XTX`` / ``XTY`` and training statistics exactly as ``training_batch`` forms them, for
        ``n_components`` = A components.  The fold's validation rows are then predicted with 1 .. A components,
        ``((x - X_mean) / X_std) @ B * Y_std + Y_mean`` (each statistic applied iff its flag is set), and scored.

        Returns a dict with ``press`` (P, A, M): the weighted sum of squared prediction errors over the validation rows,
        ``sum_w_val`` (P,): the sum of their weights (their count when unweighted), ``n_fitted`` (P,) int32: the
        components a fold could fit (a fold whose remaining ``XTY`` vanishes stops early; its later coefficients repeat
        the last ones), ``status`` (P,) int32 (``CVMX_FOLD_*`` bits) and ``B`` (P, A, K, M) with ``return_coefs``,
        else None.  ``out="torch"`` returns CUDA tensors, ``out="numpy"`` host arrays.  With ``check`` the degenerate fold
        errors of ``training_XTX_XTY`` are raised; without it such folds get NaN ``press`` / ``B`` and ``n_fitted`` 0.
        A ``UserWarning`` names folds that stopped early.

        With ``return_predictions`` the dict also holds the out-of-fold predictions the PRESS is formed from:
        ``predictions`` (n, A, M), row j the prediction of the j-th validation index of the range in CSR order (n = the
        number of stored indices of folds ``[fold_begin, fold_end)``, repeats kept) with 1 .. A components, and ``rows``
        (n,) int64, the data-set row of each (indices normalised to ``[0, N)``); without it the dict has neither key.
        A refused fold's rows are NaN; a fold that stopped early repeats its last fitted component's predictions.

        Example - root mean squared error of cross-validation per number of components and response::

            cvm.fit(X, Y); cvm.set_folds(Partitioner(folds))
            r = cvm.pls_cross_validate(20)
            rmsecv = np.sqrt(r["press"].sum(0) / r["sum_w_val"].sum())    # (20, M)

        Example - scikit-learn's ``cross_val_predict`` for every number of components (a ``Partitioner`` covers each
        row once)::

            r = cvm.pls_cross_validate(20, return_predictions=True)
            Yhat = np.empty((N, 20, M)); Yhat[r["rows"]] = r["predictions"]
        """
        self._require_fit()
        if fold_end is None:
            fold_end = self._n_folds
        if not self._has_Y:
            raise ValueError(_ERR_NO_Y)
        A, K, M, dt = int(n_components), self.K, self.M, self.dtype
        if not 1 <= A <= K:
            raise ValueError(f"n_components must be between 1 and the number of columns of X ({K}); got {A}")
        if M > 128:
            raise ValueError(f"at most 128 response columns are supported; Y has {M}")
        P = max(int(fold_end) - int(fold_begin), 0)
        n_pred = self._prediction_count(fold_begin, fold_end)
        if out == "torch":
            import torch

            tdt = torch.float64 if np.dtype(dt) == np.float64 else torch.float32
            dev = torch.device("cuda", self.device)
            press = torch.empty((P, A, M), dtype=tdt, device=dev)
            sum_w = torch.empty((P,), dtype=tdt, device=dev)
            n_fitted = torch.empty((P,), dtype=torch.int32, device=dev)
            status = torch.empty((P,), dtype=torch.int32, device=dev)
            B = torch.empty((P, A, K, M), dtype=tdt, device=dev) if return_coefs else None
            pred = torch.empty((n_pred, A, M), dtype=tdt, device=dev) if return_predictions else None
            p, mem = _tptr, _lib.DEVICE
        elif out == "numpy":
            press = np.empty((P, A, M), dt)
            sum_w = np.empty((P,), dt)
            n_fitted = np.zeros((P,), np.int32)
            status = np.zeros((P,), np.int32)
            B = np.empty((P, A, K, M), dt) if return_coefs else None
            pred = np.empty((n_pred, A, M), dt) if return_predictions else None
            p, mem = _ptr, _lib.HOST
        else:
            raise ValueError("out must be 'numpy' or 'torch'")
        with self._torch_stream() if out == "torch" else contextlib.nullcontext():
            rc = self._lib.cvmx_pls_cv_predict(self._h, int(fold_begin), int(fold_end), A, p(press), p(sum_w), p(B),
                                               p(n_fitted), p(status), p(pred), mem)
            _lib.check(rc, self._h)
        st = status.cpu().numpy() if out == "torch" else status
        if check:
            cX, cY, sX, sY = self.center_X, self.center_Y, self.scale_X, self.scale_Y
            need = (cX or cY, sX, cX or cY, sY)    # the statistics training_XTX_XTY computes
            for s in np.unique(st):
                if s:
                    self._raise_for_status(int(s), need)
        nf = n_fitted.cpu().numpy() if out == "torch" else n_fitted
        refused = (((st & _lib.FOLD_NO_NONZERO_W) != 0) & (self._flags != 0)) | (((st & _lib.FOLD_NNZ_LE_DDOF) != 0) & ((self._flags & 12) != 0))
        early = np.flatnonzero((nf < A) & ~refused)
        if early.size:
            warnings.warn(f"{early.size} fold(s) stopped before {A} components (first: fold {int(fold_begin) + int(early[0])} "
                          f"with {int(nf[early[0]])}): the remaining XTY vanished; their later coefficients repeat the last ones",
                          UserWarning, stacklevel=2)
        r = dict(press=press, sum_w_val=sum_w, n_fitted=n_fitted, status=status, B=B)
        if return_predictions:
            r.update(predictions=pred, rows=self._prediction_rows(fold_begin, fold_end, out))
        return r

    def ridge_cross_validate(self, alphas, fold_begin: int = 0, fold_end: Optional[int] = None, return_coefs: bool = False,
                             out: str = "numpy", check: bool = True, return_predictions: bool = False):
        """
        Cross-validated ridge regression over folds ``[fold_begin, fold_end)`` of the CSR (see ``set_folds``) for every
        penalty in ``alphas``, on the GPU.

        Per fold and penalty ``lam``: ``B = (XTX + lam I)^-1 XTY`` by a blocked Cholesky factorisation in float64, from the
        fold's ``XTX`` / ``XTY`` and training statistics exactly as ``training_batch`` forms them.  ``lam`` is added to the
        diagonal of the matrix as formed: with ``scale_X`` it penalises the coefficients of the standardised X columns,
        and with ``center_X`` / ``center_Y`` the intercept is not penalised (scikit-learn's ``Ridge(fit_intercept=True)``).
        The fold's validation rows are predicted as ``((x - X_mean) / X_std) @ B * Y_std + Y_mean`` (each statistic
        applied iff its flag is set) and scored.  ``alphas`` is a 1-D host sequence of 1 to 1024 finite penalties >= 0
        (repeats allowed).

        Returns a dict with ``press`` (P, L, M): the weighted sum of squared prediction errors over the validation rows,
        ``sum_w_val`` (P,): the sum of their weights (their count when unweighted), ``info`` (P, L) int32: 0, or the
        1-based column of the first pivot that was not positive (as LAPACK ``dpotrf`` reports it), ``status`` (P,) int32
        (``CVMX_FOLD_*`` bits) and ``B`` (P, L, K, M) with ``return_coefs``, else None.  A pair with ``info != 0`` gets NaN
        ``press`` / ``B``; a ``UserWarning`` counts such pairs (``lam = 0`` on a rank-deficient fold is a legitimate grid
        point, not an error).  ``out="torch"`` returns CUDA tensors, ``out="numpy"`` host arrays.  With ``check`` the
        degenerate fold errors of ``training_XTX_XTY`` are raised; without it such folds get NaN ``press`` / ``B`` for
        every penalty and ``info`` 0.

        With ``return_predictions`` the dict also holds the out-of-fold predictions the PRESS is formed from:
        ``predictions`` (n, L, M), row j the prediction of the j-th validation index of the range in CSR order (n = the
        number of stored indices of folds ``[fold_begin, fold_end)``, repeats kept) for every penalty, and ``rows``
        (n,) int64, the data-set row of each (indices normalised to ``[0, N)``); without it the dict has neither key.
        A refused fold's rows are NaN, and a pair with ``info != 0`` is NaN for that penalty only.

        Example - root mean squared error of cross-validation per penalty and response::

            cvm.fit(X, Y); cvm.set_folds(Partitioner(folds))
            r = cvm.ridge_cross_validate(np.logspace(-3, 3, 20))
            rmsecv = np.sqrt(r["press"].sum(0) / r["sum_w_val"].sum())    # (L, M)

        Example - scikit-learn's ``cross_val_predict`` for every penalty (a ``Partitioner`` covers each row once)::

            r = cvm.ridge_cross_validate(np.logspace(-3, 3, 20), return_predictions=True)
            Yhat = np.empty((N, 20, M)); Yhat[r["rows"]] = r["predictions"]
        """
        self._require_fit()
        if fold_end is None:
            fold_end = self._n_folds
        if not self._has_Y:
            raise ValueError(_ERR_NO_Y)
        if hasattr(alphas, "detach"):   # a torch tensor: the penalties are read on the host
            alphas = alphas.detach().cpu().numpy()
        try:
            lam = np.ascontiguousarray(np.asarray(alphas, dtype=np.float64))
        except (TypeError, ValueError):
            raise ValueError("alphas must be a 1-D sequence of finite penalties >= 0") from None
        if lam.ndim != 1 or not 1 <= lam.size <= 1024:
            raise ValueError(f"alphas must be a 1-D sequence of 1 to 1024 penalties; got shape {lam.shape}")
        if not (np.isfinite(lam).all() and (lam >= 0).all()):
            raise ValueError("every penalty in alphas must be finite and >= 0")
        L, K, M, dt = lam.size, self.K, self.M, self.dtype
        if M > 128:
            raise ValueError(f"at most 128 response columns are supported; Y has {M}")
        P = max(int(fold_end) - int(fold_begin), 0)
        n_pred = self._prediction_count(fold_begin, fold_end)
        if out == "torch":
            import torch

            tdt = torch.float64 if np.dtype(dt) == np.float64 else torch.float32
            dev = torch.device("cuda", self.device)
            press = torch.empty((P, L, M), dtype=tdt, device=dev)
            sum_w = torch.empty((P,), dtype=tdt, device=dev)
            info = torch.empty((P, L), dtype=torch.int32, device=dev)
            status = torch.empty((P,), dtype=torch.int32, device=dev)
            B = torch.empty((P, L, K, M), dtype=tdt, device=dev) if return_coefs else None
            pred = torch.empty((n_pred, L, M), dtype=tdt, device=dev) if return_predictions else None
            p, mem = _tptr, _lib.DEVICE
        elif out == "numpy":
            press = np.empty((P, L, M), dt)
            sum_w = np.empty((P,), dt)
            info = np.zeros((P, L), np.int32)
            status = np.zeros((P,), np.int32)
            B = np.empty((P, L, K, M), dt) if return_coefs else None
            pred = np.empty((n_pred, L, M), dt) if return_predictions else None
            p, mem = _ptr, _lib.HOST
        else:
            raise ValueError("out must be 'numpy' or 'torch'")
        with self._torch_stream() if out == "torch" else contextlib.nullcontext():
            rc = self._lib.cvmx_ridge_cv_predict(self._h, int(fold_begin), int(fold_end), _ptr(lam), L, p(press), p(sum_w),
                                                 p(B), p(info), p(status), p(pred), mem)
            _lib.check(rc, self._h)
        if check:
            st = status.cpu().numpy() if out == "torch" else status
            cX, cY, sX, sY = self.center_X, self.center_Y, self.scale_X, self.scale_Y
            need = (cX or cY, sX, cX or cY, sY)    # the statistics training_XTX_XTY computes
            for s in np.unique(st):
                if s:
                    self._raise_for_status(int(s), need)
        inf = info.cpu().numpy() if out == "torch" else info
        failed = np.argwhere(inf != 0)
        if failed.size:
            f, l = (int(x) for x in failed[0])
            warnings.warn(f"{len(failed)} (fold, penalty) pair(s) could not be factored: XTX + alpha I is not positive "
                          f"definite (first: fold {int(fold_begin) + f}, alpha {lam[l]!r} at index {l}, pivot {int(inf[f, l])}); "
                          "their press and B are NaN", UserWarning, stacklevel=2)
        r = dict(press=press, sum_w_val=sum_w, info=info, status=status, B=B)
        if return_predictions:
            r.update(predictions=pred, rows=self._prediction_rows(fold_begin, fold_end, out))
        return r

    def _prediction_count(self, fold_begin, fold_end) -> int:
        """Number of out-of-fold predictions of folds [fold_begin, fold_end): their stored CSR indices."""
        f0, f1 = int(fold_begin), int(fold_end)
        if not 0 <= f0 <= f1 <= getattr(self, "_n_folds", 0):
            return 0    # the library reports the bad range
        return int(self._offsets[f1] - self._offsets[f0])

    def _prediction_rows(self, fold_begin, fold_end, out):
        """Data-set row of every out-of-fold prediction of folds [fold_begin, fold_end): the CSR indices, normalised."""
        idx = np.asarray(self._fold_indices[self._offsets[int(fold_begin)]:self._offsets[int(fold_end)]], np.int64)
        neg = idx.size > 0 and idx.min() < 0
        if out == "torch":
            import torch

            rows = torch.from_numpy(idx).to(torch.device("cuda", self.device))
            return torch.where(rows < 0, rows + self.N, rows) if neg else rows
        return np.where(idx < 0, idx + self.N, idx) if neg else idx.copy()

    def validation_rows(self, fold: int, stats: Optional[Stats] = None, out: str = "numpy"):
        """
        ``(X[val], Y[val])`` of CSR fold number ``fold`` (see ``set_folds``) for the caller's next step - predicting the
        held-out rows.  With ``stats`` = ``(X_mean, X_std, Y_mean, Y_std)`` as returned by ``training_*`` for that fold,
        every entry that is not None is applied: ``(X[val] - X_mean) / X_std`` and likewise for Y, bit-identical to
        the numpy expressions.  ``out="torch"`` returns CUDA tensors (the rows never leave the device).
        """
        self._require_fit()
        if not 0 <= fold < getattr(self, "_n_folds", 0):
            raise ValueError(f"Fold {fold} not found.")
        K, M, dt = self.K, self.M or 0, self.dtype
        offsets = self._offsets
        n = int(offsets[fold + 1] - offsets[fold])
        apply, packed = 0, None
        if stats is not None:
            packed = np.zeros((2, K + M), dt)
            for row, lo, hi, bit, s in ((0, 0, K, 1, stats[0]), (1, 0, K, 4, stats[1]), (0, K, K + M, 2, stats[2]), (1, K, K + M, 8, stats[3])):
                if s is not None and hi > lo:
                    packed[row, lo:hi] = np.asarray(s, dtype=dt).reshape(-1)
                    apply |= bit
        if out == "torch":
            import torch

            tdt = torch.float64 if np.dtype(dt) == np.float64 else torch.float32
            dev = torch.device("cuda", self.device)
            Xv = torch.empty((n, K), dtype=tdt, device=dev)
            Yv = torch.empty((n, M), dtype=tdt, device=dev) if M else None
            st = torch.from_numpy(packed).to(dev) if apply else None
            torch.cuda.current_stream(dev).synchronize()
            p = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
            rc = self._lib.cvmx_validation_rows(self._h, fold, p(st), apply, p(Xv), p(Yv), _lib.DEVICE)
            _lib.check(rc, self._h)
            self.sync()
            return Xv, Yv
        if out != "numpy":
            raise ValueError("out must be 'numpy' or 'torch'")
        Xv = np.empty((n, K), dt)
        Yv = np.empty((n, M), dt) if M else None
        rc = self._lib.cvmx_validation_rows(self._h, fold, _ptr(packed) if apply else None, apply, _ptr(Xv), _ptr(Yv), _lib.HOST)
        _lib.check(rc, self._h)
        return Xv, Yv

    def _pinned(self, name: str, shape, dtype=None) -> np.ndarray:
        import torch

        dtype = np.dtype(self.dtype if dtype is None else dtype)
        pool = self.__dict__.setdefault("_pinned_pool", {})
        need = int(np.prod(shape)) * dtype.itemsize
        buf = pool.get(name)
        if buf is None or buf.numel() < need:
            buf = pool[name] = torch.empty((max(need, 1),), dtype=torch.uint8, pin_memory=True)
        return buf.numpy()[:need].view(dtype).reshape(shape)

    def sync(self) -> None:
        _lib.check(self._lib.cvmx_sync(self._h), self._h)

    def set_scan_mode(self, mode: int) -> None:
        """How float64 column sums in numpy's sequential order are evaluated (include/cvmx.h, cvmx_set_scan_mode):
        0 dependent-add chains only, 1 (default) the bit-identical binade scan when the chains are on the critical
        path, 2 the scan whenever a fold has >= 1024 rows."""
        _lib.check(self._lib.cvmx_set_scan_mode(self._h, int(mode)), self._h)

    def set_loo_mode(self, mode: int) -> None:
        """Leave-one-out / leave-few-out batches (include/cvmx.h, cvmx_set_loo_mode): 0 (default) streaming form, matrices
        within ~1e-15 of the reference; 1 exact form, matrices bit-identical to the reference for one-row folds."""
        _lib.check(self._lib.cvmx_set_loo_mode(self._h, int(mode)), self._h)

    @property
    def folds_cached(self) -> bool:
        """True while the fold Grams kept by ``fit(..., folds=...)`` serve ``training_batch``."""
        return bool(self._lib.cvmx_folds_are_cached(self._h))

    @property
    def scan_launch_count(self) -> int:
        return int(self._lib.cvmx_scan_launch_count(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._lib.cvmx_launch_count(self._h))
