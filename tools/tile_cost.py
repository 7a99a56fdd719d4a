#!/usr/bin/env python
"""Relative cost of a diagonal Gram tile, the constant of the row-split plan (plan_tapered in cvmx_api.cu).

    python tools/tile_cost.py --out DIR [--rows 2000000] [--steps 20] [--reps 3]

K = 128, M = 128 (float64, weighted, centre + scale, 5 folds, inputs generated on the device from seed 42), so a fold
has exactly one tile of each kind: training_batch with only XTX runs the diagonal tile (0, 0) alone and with only XTY
the off-diagonal tile (0, 1) alone, over the same row-split units.  Both take k_gram's time from the library's own
CUDA events (cvmx_profile_read) over `steps` calls, alternating `reps` times; the ratio diagonal / off-diagonal is
the cost a diagonal tile is given in the plan.  Writes DIR/tile_cost.json and prints it.
"""

from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rows", type=int, default=2_000_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()

    import torch

    from cvmatrix_b200 import CVMatrix, Partitioner, _lib

    N, K, M, P = a.rows, 128, 128, 5
    g = torch.Generator(device="cuda").manual_seed(42)
    m = CVMatrix()
    block = 100_000
    m.fit_begin(N, K, M, weighted=True, max_block_rows=block)
    for r0 in range(0, N, block):
        n = min(block, N - r0)
        X = torch.rand((n, K), generator=g, device="cuda", dtype=torch.float64)
        Y = torch.rand((n, M), generator=g, device="cuda", dtype=torch.float64)
        w = torch.rand((n,), generator=g, device="cuda", dtype=torch.float64)
        torch.cuda.synchronize()
        m.fit_rows(r0, X, Y, w)
    m.fit_end()
    m.set_folds(Partitioner(np.arange(N) % P))

    def gram_ms(xtx: bool) -> float:
        run = lambda: m.training_batch(return_XTX=xtx, return_XTY=not xtx, out="torch")  # noqa: E731
        run()   # warm-up, plan and scratch
        torch.cuda.synchronize()
        ms, n = (C.c_double * 3)(), (C.c_int64 * 3)()
        _lib.check(m._lib.cvmx_profile_read(m._h, ms, n), m._h)   # reset
        _lib.check(m._lib.cvmx_profile_enable(m._h, 1), m._h)
        for _ in range(a.steps):
            run()
        _lib.check(m._lib.cvmx_profile_read(m._h, ms, n), m._h)
        _lib.check(m._lib.cvmx_profile_enable(m._h, 0), m._h)
        return ms[1] / a.steps

    diag, off = [], []
    for _ in range(a.reps):
        diag.append(gram_ms(True))
        off.append(gram_ms(False))
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    res = dict(
        device=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip() or q.stderr.strip(),
        shape=dict(N=N, K=K, M=M, P=P, dtype="float64"), steps=a.steps,
        k_gram_ms_diagonal_tile=diag, k_gram_ms_offdiagonal_tile=off,
        ratio_per_rep=[d / o for d, o in zip(diag, off)],
        ratio_median=statistics.median(d / o for d, o in zip(diag, off)),
    )
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "tile_cost.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
