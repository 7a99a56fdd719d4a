#!/usr/bin/env python
"""Cross-validated ridge regression on the GPU (CVMatrix.ridge_cross_validate) against the fold path it builds on.

    python tools/bench_ridge.py --out DIR [--cases cfg2,cfg3,cfg4,cfg5s] [--reps 3] [--penalties 20] [--predictions]

Per case: inputs are generated on the device (uniform [0, 1), seed 42, weighted) and fitted through fit_begin /
fit_rows / fit_end, the folds are arange(N) % P, the penalties are L log-spaced values over 1e-3 .. 1e3 times
trace(XTX) / K of the first fold.  Timed with CUDA events on the same range and resident inputs:
``training_batch(out="torch")`` (XTX, XTY and statistics of every fold) and ``ridge_cross_validate(alphas,
out="torch")`` (the same matrices into library scratch, then the factorisations, substitutions and PRESS); the
difference is the cost of ridge + PRESS.  A separate run under torch.profiler gives the time of every kernel.  The flop
model counts P L K^3 / 3 for the factorisations, 2 P L K^2 M for the substitutions and 2 n_val K L M for PRESS; the
achieved FP64 rate of the factorisation is its flops over the summed time of k_ridge_potrf_diag, k_ridge_trsm and
k_ridge_syrk.  The device name and power limit are read in the same run.  With --predictions the same call is also
timed with ``return_predictions=True`` (out="torch"), alternating with the plain call, and the difference is reported
beside the HBM bound of writing n * L * M * sizeof(T) bytes of predictions.  Writes DIR/bench_ridge.json (and one line
per case to stdout).

Cases (float64, center + scale X and Y):
  cfg2   N = 1,000,000  K = 500   M = 10   P = 5
  cfg3   N = 1,000,000  K = 500   M = 10   P = 1000
  cfg4   N = 20,000     K = 500   M = 10   P = 20,000 (leave-one-out)
  cfg5s  N = 400,000    K = 5000  M = 100  P = 10     (cfg 5 shape at a fifth of its rows)
"""

from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_pls import CASES, device_info, make_model, predictions_overhead, timed  # noqa: E402

FACTOR_KERNELS = ("k_ridge_potrf_diag", "k_ridge_trsm", "k_ridge_syrk")


def kernel_times(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        if t and ("k_" in ev.key or "Memcpy" in ev.key or "Memset" in ev.key):
            out[ev.key[:120]] = {"ms": t / 1e3, "calls": ev.count}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["ms"]))


def flop_model(N, K, M, P, L):
    return {"factorisation": P * L * K**3 / 3, "substitutions": 2 * P * L * K**2 * M, "press": 2 * N * K * L * M}


def run_case(name, L, reps, predictions=False):
    import torch

    c = CASES[name]
    N, K, M, P = c["N"], c["K"], c["M"], c["P"]
    m = make_model(N, K, M, P)
    XTX0 = m.training_batch(0, 1, return_XTY=False, out="torch")["XTX"][0]
    alphas = np.logspace(-3, 3, L) * float(torch.trace(XTX0)) / K
    del XTX0
    tb = lambda: m.training_batch(out="torch", check=False)  # noqa: E731
    ridge = lambda: m.ridge_cross_validate(alphas, out="torch", check=False)  # noqa: E731
    t_tb = timed(tb, reps)
    t_ridge = timed(ridge, reps)
    r = m.ridge_cross_validate(alphas, out="torch")
    rmsecv = torch.sqrt(r["press"].sum(0) / r["sum_w_val"].sum()).cpu().numpy()
    n_failed = int((r["info"] != 0).sum())
    kern = kernel_times(ridge)
    diff = float(np.median(t_ridge) - np.median(t_tb))
    flops = flop_model(N, K, M, P, L)
    fact_ms = sum(v["ms"] for k, v in kern.items() if any(n in k for n in FACTOR_KERNELS))
    out = dict(
        case=name, N=N, K=K, M=M, P=P, L=L, dtype="float64",
        training_batch_ms=t_tb, ridge_cross_validate_ms=t_ridge,
        ridge_plus_press_ms=diff,
        flops=flops,
        factorisation_kernels_ms=fact_ms,
        factorisation_TFLOPs=flops["factorisation"] / (fact_ms * 1e-3) / 1e12 if fact_ms else None,
        kernels=kern,
        failed_pairs=n_failed,
        best_penalty_index=[int(i) for i in np.argmin(rmsecv, axis=0)[:3]],
    )
    del r
    if predictions:
        pred = lambda: m.ridge_cross_validate(alphas, out="torch", check=False, return_predictions=True)  # noqa: E731
        out["predictions"] = predictions_overhead(ridge, pred, reps, N * L * M * 8)
        out["predictions"]["kernels"] = kernel_times(pred)
    del m
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_ridge.json (created if missing)")
    ap.add_argument("--cases", default="cfg2,cfg3,cfg4,cfg5s")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--penalties", type=int, default=20)
    ap.add_argument("--predictions", action="store_true", help="also time return_predictions=True against the plain call")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_ridge.py needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    res = {"device": device_info(), "cases": []}
    for name in a.cases.split(","):
        r = run_case(name, a.penalties, a.reps, a.predictions)
        res["cases"].append(r)
        print(json.dumps({k: v for k, v in r.items() if k != "kernels"}), flush=True)
    res["device_after"] = device_info()
    with open(os.path.join(a.out, "bench_ridge.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
