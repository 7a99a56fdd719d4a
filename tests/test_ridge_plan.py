"""CPU tests of cvmx_ridge_plan, the host-only launch plan of cross-validated ridge (no CUDA call): at shapes up to
K = 5000, M = 128, L = 1024 and P = 20,000, every grid and shared-memory size is inside the device limits, the scratch
arrays end inside the reserved bytes, the pass stays within the ~1 GiB rule, windows and passes cover the folds and
penalties exactly once, and a shape that cannot fit is reported as infeasible rather than clipped."""

import ctypes as C
import itertools

import numpy as np
import pytest

BUDGET = 1 << 30
MAX_SMEM = 227 * 1024
MAX_X, MAX_Y = 2**31 - 1, 65535


def _plan(K, M, L, P, dtype=1, mem=0, want_B=1):
    from cvmatrix_b200 import _lib, build

    build.build_lib()
    plan = np.zeros(_lib.RIDGE_PLAN_LEN, np.int64)
    rc = _lib.load().cvmx_ridge_plan(K, M, L, P, dtype, mem, want_B, plan.ctypes.data_as(C.c_void_p))
    return rc, plan


SHAPES = [(1, 1, 1, 0), (1, 1, 1, 1), (10, 2, 3, 5), (63, 1, 20, 7), (64, 3, 20, 1000), (65, 40, 20, 1000), (300, 128, 1024, 20),
          (500, 10, 20, 1000), (500, 10, 20, 20_000), (500, 128, 1024, 20_000), (2000, 64, 100, 50), (5000, 100, 20, 10),
          (5000, 128, 1024, 20_000), (4999, 1, 1, 1)]


@pytest.mark.parametrize("K,M,L,P", SHAPES)
@pytest.mark.parametrize("mem,want_B,dtype", list(itertools.product((0, 1), (0, 1), (0, 1))))
def test_plan_within_limits_and_covers(K, M, L, P, mem, want_B, dtype):
    from cvmatrix_b200 import _lib

    rc, p = _plan(K, M, L, P, dtype, mem, want_B)
    assert rc == _lib.OK and p[_lib.RIDGE_FEASIBLE] == 1
    W, Lp = int(p[_lib.RIDGE_FOLDS_PER_WINDOW]), int(p[_lib.RIDGE_PENALTIES_PER_PASS])
    assert 1 <= W <= max(P, 1) and 1 <= Lp <= L
    # a pass is every penalty of its window, or one fold: its outputs are one contiguous range
    assert Lp == L or W == 1
    # scratch: ends increase, all inside the reserved bytes; the pass stays within the window rule (one pair always allowed)
    ends = p[_lib.RIDGE_END_A:_lib.RIDGE_END_STATUS + 1]
    assert (np.diff(ends) >= 0).all() and ends[-1] == p[_lib.RIDGE_SCRATCH_BYTES]
    pair_mat = (K + M) * K * 8
    assert p[_lib.RIDGE_END_A] >= W * Lp * pair_mat
    assert p[_lib.RIDGE_SCRATCH_BYTES] <= BUDGET or (W == 1 and Lp == 1)
    assert p[_lib.RIDGE_PART_BYTES] <= 256 << 20 or p[_lib.RIDGE_CHUNKS_PER_LAUNCH] == 1
    assert p[_lib.RIDGE_CHUNKS_PER_LAUNCH] >= 1
    # grids and dynamic shared memory
    for k in range(_lib.RK_COUNT):
        gx, gy = p[_lib.RIDGE_GRID + 2 * k], p[_lib.RIDGE_GRID + 2 * k + 1]
        assert 0 <= gx <= MAX_X and 0 <= gy <= MAX_Y, _lib.RIDGE_KERNELS[k]
        assert 0 <= p[_lib.RIDGE_SMEM + k] <= MAX_SMEM, _lib.RIDGE_KERNELS[k]
    assert p[_lib.RIDGE_GRID + 2 * _lib.RK_COEFS] == (W * Lp if want_B else 0)
    # the trailing update of the first panel is the largest: pairs x lower tiles
    nb0 = min(64, K)
    if K > nb0:
        R, Cc = -(-(K + M - nb0) // 64), -(-(K - nb0) // 64)
        assert p[_lib.RIDGE_GRID + 2 * _lib.RK_SYRK] == W * Lp * (Cc * (Cc + 1) // 2 + (R - Cc) * Cc)
    # windows and passes cover the fold range and the penalty list exactly once
    seen = np.zeros((max(P, 0), L), np.int32)
    for c0 in range(0, P, W):
        for l0 in range(0, L, Lp):
            seen[c0:c0 + W, l0:l0 + Lp] += 1
    assert (seen == 1).all()


def test_both_splits_occur():
    from cvmatrix_b200 import _lib

    # the shape tests/test_gpu_ridge.py uses to cross windows and passes
    rc, p = _plan(400, 2, 1024, 3)
    assert rc == _lib.OK and p[_lib.RIDGE_FOLDS_PER_WINDOW] == 1 and 1 < p[_lib.RIDGE_PENALTIES_PER_PASS] < 1024
    rc, p = _plan(300, 2, 1024, 3)
    assert rc == _lib.OK and p[_lib.RIDGE_FOLDS_PER_WINDOW] == 1 and p[_lib.RIDGE_PENALTIES_PER_PASS] == 1024


def test_splits_of_the_edge_shapes():
    from cvmatrix_b200 import _lib

    # the shapes tests/test_gpu_cv_edges.py uses, for host and device outputs, with and without B
    for mem, want_B in itertools.product((0, 1), (0, 1)):
        # PRESS over several launches: 131,072 columns leave 255 chunks per launch; two folds of 313 chunks need three
        rc, p = _plan(4, 128, 1024, 2, mem=mem, want_B=want_B)
        assert rc == _lib.OK and p[_lib.RIDGE_FOLDS_PER_WINDOW] == 2 and p[_lib.RIDGE_PENALTIES_PER_PASS] == 1024
        assert p[_lib.RIDGE_CHUNKS_PER_LAUNCH] == 255
        # leave-one-out over 595 folds: three to five windows of all 16 penalties
        rc, p = _plan(200, 8, 16, 595, mem=mem, want_B=want_B)
        W = p[_lib.RIDGE_FOLDS_PER_WINDOW]
        assert rc == _lib.OK and p[_lib.RIDGE_PENALTIES_PER_PASS] == 16 and 3 <= -(-595 // W) <= 5
        # one fold per window, its penalties in passes
        rc, p = _plan(400, 2, 1024, 3, mem=mem, want_B=want_B)
        assert rc == _lib.OK and p[_lib.RIDGE_FOLDS_PER_WINDOW] == 1 and 1 < p[_lib.RIDGE_PENALTIES_PER_PASS] < 1024


def test_infeasible_and_invalid_shapes():
    from cvmatrix_b200 import _lib

    # one pair of K = 65,000 columns is ~34 GB: reported as infeasible, not clipped to a smaller pass
    rc, p = _plan(65_000, 1, 1, 1)
    assert rc == _lib.ERR_INVALID and p[_lib.RIDGE_FEASIBLE] == 0
    assert p[_lib.RIDGE_FOLDS_PER_WINDOW] == 1 and p[_lib.RIDGE_PENALTIES_PER_PASS] == 1
    assert p[_lib.RIDGE_SCRATCH_BYTES] >= 65_001 * 65_000 * 8
    for bad in [(0, 1, 1, 1), (10, 0, 1, 1), (10, 129, 1, 1), (10, 1, 0, 1), (10, 1, 1025, 1), (10, 1, 1, -1)]:
        rc, p = _plan(*bad)
        assert rc == _lib.ERR_INVALID and p[_lib.RIDGE_FEASIBLE] == 0, bad
    assert _plan(10, 1, 1, 1, dtype=2)[0] == _lib.ERR_INVALID
    assert _plan(10, 1, 1, 1, mem=2)[0] == _lib.ERR_INVALID
