#!/usr/bin/env python
"""Cross-validated PLS on the GPU (CVMatrix.pls_cross_validate) against the fold path it builds on.

    python tools/bench_pls.py --out DIR [--cases cfg2,cfg3,cfg4,cfg5s] [--reps 3] [--components 20] [--predictions]

Per case: inputs are generated on the device (uniform [0, 1), seed 42, weighted) and fitted through fit_begin /
fit_rows / fit_end, the folds are arange(N) % P.  Timed with CUDA events on the same range and resident inputs:
``training_batch(out="torch")`` (XTX, XTY and statistics of every fold) and ``pls_cross_validate(A, out="torch")``
(the same matrices into library scratch, then IKPLS and PRESS); the difference is the cost of PLS + PRESS.  A separate
run under torch.profiler gives the time of every kernel.  Bytes follow DESIGN.md's model: A * P * K^2 * sizeof(T)
for the XTX r products plus one read of the validation rows (K + M values each) for PRESS; the share of the HBM bound
is (bytes / 7.7 TB/s) over the PLS + PRESS time.  The CPU figure is the numpy oracle (oracle/pls_oracle.py) timed on
the engine's own matrices and validation rows for the first `cpu_folds` folds of the case, reported as such.
With --predictions the same call is also timed with ``return_predictions=True`` (out="torch"), alternating with the
plain call in one loop, and the difference is reported beside the HBM bound of writing n * A * M * sizeof(T) bytes of
predictions (n = N: the folds partition the rows).  Writes DIR/bench_pls.json (and one line per case to stdout).

Cases (A = 20 components, float64, center + scale X and Y):
  cfg2   N = 1,000,000  K = 500   M = 10   P = 5
  cfg3   N = 1,000,000  K = 500   M = 10   P = 1000
  cfg4   N = 20,000     K = 500   M = 10   P = 20,000 (leave-one-out)
  cfg5s  N = 400,000    K = 5000  M = 100  P = 10     (cfg 5 shape at a fifth of its rows)
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

CASES = {
    "cfg2": dict(N=1_000_000, K=500, M=10, P=5, cpu_folds=1),
    "cfg3": dict(N=1_000_000, K=500, M=10, P=1000, cpu_folds=10),
    "cfg4": dict(N=20_000, K=500, M=10, P=20_000, cpu_folds=100),
    "cfg5s": dict(N=400_000, K=5000, M=100, P=10, cpu_folds=1),
}
HBM_BPS = 7.7e12   # HGX B200 data sheet, one GPU


def device_info():
    import torch

    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def make_model(N, K, M, P):
    import torch

    from cvmatrix_b200 import CVMatrix, Partitioner

    g = torch.Generator(device="cuda").manual_seed(42)
    m = CVMatrix()
    block = 50_000
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
    return m


def timed(fn, reps):
    import torch

    fn()   # warm-up: module load, scratch allocation
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def predictions_overhead(plain, with_pred, reps, pred_bytes):
    """Median CUDA-event times of `plain` and `with_pred`, alternated in one loop after a warm-up of each, their
    difference, and the HBM bound of writing the predictions."""
    plain(), with_pred()
    tp, tw = [], []
    for _ in range(reps):
        tp += timed_once(plain)
        tw += timed_once(with_pred)
    d = float(np.median(tw) - np.median(tp))
    return dict(plain_ms=tp, with_predictions_ms=tw, overhead_ms=d,
                overhead_share=d / float(np.median(tp)), prediction_bytes=pred_bytes,
                prediction_write_hbm_bound_ms=pred_bytes / HBM_BPS * 1e3)


def timed_once(fn):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return [e0.elapsed_time(e1)]


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
        if t and ("k_" in ev.key or "Memcpy" in ev.key):
            out[ev.key[:120]] = {"ms": t / 1e3, "calls": ev.count}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["ms"]))


def cpu_oracle(m, A, n):
    import pls_oracle as po

    tb = m.training_batch(0, n)
    t0 = time.perf_counter()
    for f in range(n):
        B, _ = po.ikpls(tb["XTX"][f], tb["XTY"][f], A)
        Xv, Yv = m.validation_rows(f)
        wv = np.ones(len(Xv))   # timing only: the weights do not change the work
        po.press(Xv, Yv, wv, B, tb["X_mean"][f], tb["X_std"][f], tb["Y_mean"][f], tb["Y_std"][f])
    return (time.perf_counter() - t0) * 1e3


def run_case(name, A, reps, predictions=False):
    import torch

    c = CASES[name]
    N, K, M, P = c["N"], c["K"], c["M"], c["P"]
    m = make_model(N, K, M, P)
    tb = lambda: m.training_batch(out="torch", check=False)  # noqa: E731
    pls = lambda: m.pls_cross_validate(A, out="torch", check=False)  # noqa: E731
    t_tb = timed(tb, reps)
    t_pls = timed(pls, reps)
    r = m.pls_cross_validate(A, out="torch")
    rmsecv = torch.sqrt(r["press"].sum(0) / r["sum_w_val"].sum()).cpu().numpy()
    kern = kernel_times(pls)
    diff = float(np.median(t_pls) - np.median(t_tb))
    n_val = N   # the folds partition the rows: every row is read once by PRESS
    bytes_prod = A * P * K * K * 8
    bytes_press = n_val * (K + M) * 8
    xtx_ms = sum(v["ms"] for k, v in kern.items() if "k_pls_xtx_r" in k)
    out = dict(
        case=name, N=N, K=K, M=M, P=P, A=A, dtype="float64",
        training_batch_ms=t_tb, pls_cross_validate_ms=t_pls,
        pls_plus_press_ms=diff,
        model_bytes={"xtx_r_products": bytes_prod, "press_rows": bytes_press},
        hbm_bound_ms=(bytes_prod + bytes_press) / HBM_BPS * 1e3,
        hbm_share_of_pls_plus_press=((bytes_prod + bytes_press) / HBM_BPS * 1e3) / diff if diff > 0 else None,
        k_pls_xtx_r_ms=xtx_ms,
        k_pls_xtx_r_GBps=bytes_prod / (xtx_ms * 1e-3) / 1e9 if xtx_ms else None,
        kernels=kern,
        n_fitted_min=int(r["n_fitted"].min()),
        rmsecv_first_component=[float(x) for x in rmsecv[0][:3]],
        cpu_oracle={"folds": c["cpu_folds"], "ms": cpu_oracle(m, A, c["cpu_folds"]),
                    "what": "oracle/pls_oracle.py IKPLS + PRESS on the engine's XTX / XTY / statistics / validation rows, "
                            "first folds only, host numpy"},
    )
    if predictions:
        pred = lambda: m.pls_cross_validate(A, out="torch", check=False, return_predictions=True)  # noqa: E731
        out["predictions"] = predictions_overhead(pls, pred, reps, N * A * M * 8)
        out["predictions"]["kernels"] = kernel_times(pred)
    del m
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_pls.json (created if missing)")
    ap.add_argument("--cases", default="cfg2,cfg3,cfg4,cfg5s")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--components", type=int, default=20)
    ap.add_argument("--predictions", action="store_true", help="also time return_predictions=True against the plain call")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_pls.py needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    res = {"device": device_info(), "cases": []}
    for name in a.cases.split(","):
        r = run_case(name, a.components, a.reps, a.predictions)
        res["cases"].append(r)
        print(json.dumps({k: v for k, v in r.items() if k != "kernels"}, default=str), flush=True)
    res["device_after"] = device_info()
    with open(os.path.join(a.out, "bench_pls.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
