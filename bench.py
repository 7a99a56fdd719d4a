#!/usr/bin/env python
"""
bench.py - fold matrices / second of the cvmatrix hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2|cfg3|cfg4|cfg5s] [--impl native|reference]
                    [--dump-outputs DIR]

One "step" = one pass of the batched fold path (cvmx_training_batch: weight masses, numpy-order
moments, DMMA Gram downdate, fused centering/scaling epilogue) over ALL folds of the workload, inputs
resident in HBM, outputs written to HBM.  `value` = folds processed by all ranks / max-over-ranks device
time.  `e2e` = the reference benchmark's own definition (benchmarks/benchmark.py:52-158): Partitioner +
fit (host->device copy of X, Y, w from pinned memory) + all folds + device->host copy of every result,
through the public CVMatrix API.  `cpu_baseline` / `--impl reference` time the reference itself - the
unmodified package staged in oracle/_ref by `make -C oracle ref` (kind "reference"), else the pinned numpy
restatement oracle/cvmatrix_oracle.py (kind "port") - on the box's host cores, all BLAS threads.
`parity` compares the timed path's results with that reference on the same inputs (relative Frobenius error
of XTX, XTY and the joint [XTX | XTY]; statistics bit for bit), `also` carries device-timed lines of the other
two single-GPU workloads (cfg3, cfg4) measured in the same process.  `--dump-outputs DIR` writes the results of the
last timed step to DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for output.

Workloads (BASELINE.json configs; inputs per benchmarks/benchmark.py:223-232, seed 42, uniform [0,1)):
  cfg2  N=1,000,000 K=500 M=10 float64 weighted center+scale, 5 folds      (default; metric config)
  cfg3  same data, 1,000 folds
  cfg4  leave-one-out N=20,000 K=500 M=10 (20,000 folds)
Inputs (4.09 GB) are far larger than the 126 MB L2, so consecutive steps cannot reuse cached inputs.
"""

from __future__ import annotations

import os
import sys


def _host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        return os.cpu_count() or 1


# The CPU reference must get every host core: torchrun exports OMP_NUM_THREADS=1 to its workers, which would
# starve OpenBLAS on rank 0 (the only rank that runs the reference).  Fixed before numpy loads its BLAS.
if int(os.environ.get("RANK", "0")) == 0:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        if os.environ.get(_v, "") in ("", "1"):
            os.environ[_v] = str(_host_cores())

import argparse  # noqa: E402
import ctypes as C  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    "cfg2": dict(N=1_000_000, K=500, M=10, P=5, name="N=1M K=500 M=10 f64 weighted center+scale 5-fold"),
    "cfg3": dict(N=1_000_000, K=500, M=10, P=1000, name="N=1M K=500 M=10 f64 weighted center+scale 1000-fold"),
    "cfg4": dict(N=20_000, K=500, M=10, P=20_000, name="LOO N=20k K=500 M=10 f64 weighted center+scale"),
    # contract self-test shape (tests/test_bench_contract.py)
    "tiny": dict(N=4_000, K=24, M=3, P=4, name="self-test: N=4k K=24 M=3 f64 4-fold"),
    # cfg 5 (wide, K=5000 M=100) at reduced N: the full N=2M matrix is 80 GB and cannot be generated on the host
    "cfg5s": dict(N=100_000, K=5000, M=100, P=10, name="wide K=5000 M=100 f64 weighted center+scale 10-fold at N=100k (cfg 5 scaled to 1/20 of its rows)"),
    # cfg 5 at FULL size: the rows are produced block by block on the device and sharded across the GPUs (row-slab mode)
    "cfg5": dict(N=2_000_000, K=5000, M=100, P=10, device_generated=True,
                 name="wide N=2M K=5000 M=100 f64 weighted center+scale 10-fold, rows generated on the device and sharded across the GPUs"),
    "cfg5f32": dict(N=2_000_000, K=5000, M=100, P=10, device_generated=True, f32=True,
                    name="wide N=2M K=5000 M=100 f32 weighted center+scale 10-fold, rows generated on the device and sharded across the GPUs"),
    # reduced shapes for ncu captures only (same per-CTA work as cfg2 / cfg3 / cfg4, fewer CTAs)
    "prof2": dict(N=200_000, K=500, M=10, P=5, name="profiling: N=200k K=500 M=10 f64 5-fold"),
    "prof3": dict(N=200_000, K=500, M=10, P=200, name="profiling: N=200k K=500 M=10 f64 200-fold"),
    "prof4": dict(N=2_000, K=500, M=10, P=2_000, name="profiling: LOO N=2k K=500 M=10 f64"),
}
METRIC = "fold matrices/sec"
UNIT = "fold-matrices/s"
REF_BUDGET_S = 150.0   # wall-clock budget that bounds the reference arm's warm-up steps


def fp64_peak_tflops():
    """Measured DMMA.8x8x4 issue-rate peak on this pool's B200 (tools/ubench_fp64.cu ->
    profiles/r01_fp64_calibration.json); MEASURED_PEAKS.json carries no FP64 figure."""
    try:
        with open(os.path.join(ROOT, "profiles", "r01_fp64_calibration.json")) as f:
            d = json.load(f)
        return float(d["dmma_tflops_bps2_w16_acc16"]), "measured DMMA.8x8x4 peak (profiles/r01_fp64_calibration.json)"
    except Exception:
        return 37.0, "fallback: nominal B200 FP64 37 TFLOP/s"


def hbm_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def make_host_inputs(cfg, pinned):
    """Seeded synthetic inputs written straight into (optionally pinned) host buffers."""
    N, K, M, P = cfg["N"], cfg["K"], cfg["M"], cfg["P"]
    rng = np.random.default_rng(42)
    if pinned:
        import torch

        Xt = torch.empty((N, K), dtype=torch.float64, pin_memory=True)
        Yt = torch.empty((N, M), dtype=torch.float64, pin_memory=True)
        wt = torch.empty((N,), dtype=torch.float64, pin_memory=True)
        X, Y, w = Xt.numpy(), Yt.numpy(), wt.numpy()
        keep = (Xt, Yt, wt)
    else:
        X, Y, w = np.empty((N, K)), np.empty((N, M)), np.empty(N)
        keep = None
    rng.random(out=X)
    rng.random(out=Y)
    rng.random(out=w)
    folds = np.arange(N) % P
    return X, Y, w, folds, keep


def row_sharded_mode(P, world):
    return world > 1 and P < 4 * world          # cvmatrix_b200.sharding.use_row_sharding


def config_dict(cfg, world):
    """The `config` object of the JSON line - identical for the native and the reference arm."""
    N, K, M, P = cfg["N"], cfg["K"], cfg["M"], cfg["P"]
    if cfg.get("device_generated"):
        return {"workload": cfg["name"], "N": N, "K": K, "M": M, "folds": P,
                "parallelism": f"rows of the data set sharded x{world} (row slabs): chained column sums, per-slab Grams summed by the fold owners over NVLink peer memory",
                "l2_policy": "inputs (82 GB float64) far larger than L2; no flush needed",
                "step": "batched fold path over all folds, inputs resident in HBM, outputs to HBM"}
    par = (f"rows of each fold sharded x{world}, fold owners reduce over NVLink peer memory" if row_sharded_mode(P, world)
           else f"fold-sharded x{world}")
    return {"workload": cfg["name"], "N": N, "K": K, "M": M, "folds": P, "parallelism": par,
            "l2_policy": ("inputs (4.09 GB) larger than L2; no flush needed" if N * K * 8 > 2e8
                          else ("inputs smaller than L2 (LOO): outputs (>=8 GB per step) stream through L2" if P > 1000
                                else "self-test shape: inputs smaller than L2")),
            "step": "batched fold path over all folds, inputs resident in HBM, outputs to HBM"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        busy = [s for s in sm if s > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU reference (checker / baseline only)
# ---------------------------------------------------------------------------------------------------------------
def load_reference():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference_loader

    threads = reference_loader.use_all_host_threads()
    RefCV, RefPart, kind = reference_loader.load()
    return RefCV, RefPart, kind, threads, reference_loader.blas_threads()


def rel_fro(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    nb = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / nb) if nb > 0 else float(np.linalg.norm(a - b))


def parity_entry(got, ref):
    """got / ref: (XTX, XTY, (X_mean, X_std, Y_mean, Y_std)) of one fold."""
    XTX, XTY, st = got
    rXTX, rXTY, rst = ref
    exact = all((a is None and b is None) or (a is not None and b is not None and np.array_equal(np.asarray(a).reshape(-1), np.asarray(b).reshape(-1)))
                for a, b in zip(st, rst))
    return {"xtx": rel_fro(XTX, rXTX), "xty": rel_fro(XTY, rXTY),
            "joint": rel_fro(np.hstack([XTX, XTY]), np.hstack([rXTX, rXTY])), "stats_bit_exact": bool(exact)}


def parity_summary(entries, kind, what):
    if not entries:
        return None
    return {"xtx": max(e["xtx"] for e in entries), "xty": max(e["xty"] for e in entries), "joint": max(e["joint"] for e in entries),
            "stats_bit_exact": all(e["stats_bit_exact"] for e in entries), "folds_checked": len(entries),
            "against": f"{kind} (numpy backend) on the same inputs", "what": what,
            "tolerance": "north_star: relFro <= 1e-12 (float64); centred XTY alone at N = 1M has a ~3-4e-12 floor against OpenBLAS for "
                         "any independent summation order (SURVEY.md Appendix B), XTX and the joint matrix do not"}


def run_reference(args, cfg, rank, world):
    """Reference arm: the reference's own CPU implementation at FULL size, all host threads; one step =
    Partitioner + fit + every fold (training_XTX_XTY), exactly what benchmarks/benchmark.py:52-158 times.  Exactly
    --steps steps are timed; warm-up steps after the first run only while they fit REF_BUDGET_S (their count is printed)."""
    if rank != 0:
        return
    RefCV, RefPart, kind, threads, blas = load_reference()
    N, K, M, P = cfg["N"], cfg["K"], cfg["M"], cfg["P"]
    row_scale = 1.0
    if cfg.get("device_generated"):
        # the full matrix (80 GB; X, WX, sq_X would need 240 GB of host memory) cannot exist on the host: time 1/50 of
        # the rows and scale linearly in N (every term of the reference's cost is linear in N at fixed K, M, P)
        row_scale = 50.0
        cfg = dict(cfg, N=int(N / row_scale))
        N = cfg["N"]
    X, Y, w, folds, _ = make_host_inputs(cfg, pinned=False)
    if cfg.get("f32"):
        X, Y, w = X.astype(np.float32), Y.astype(np.float32), w.astype(np.float32)
    ref_dtype = np.float32 if cfg.get("f32") else np.float64
    loo = P > 1000
    # leave-one-out at full size is ~90 s per pass: time the full fit and a fixed sample of folds per step
    n_folds = P if not loo else 2000

    def one_step():
        t0 = time.perf_counter()
        part = RefPart(folds)
        m = RefCV(dtype=ref_dtype, copy=False)
        m.fit(X, Y, w)
        t1 = time.perf_counter()
        for f in list(part.folds_dict)[:n_folds]:
            m.training_XTX_XTY(part.get_validation_indices(f))
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1

    t_begin = time.perf_counter()
    first = one_step()                      # warm-up step 1 (also the calibration of the clamp)
    est = sum(first)
    warmup = 1
    while warmup < args.warmup and (time.perf_counter() - t_begin) + est * 2 < REF_BUDGET_S * 0.4:
        one_step()
        warmup += 1
    steps = args.steps
    t_fit = t_fold = 0.0
    for _ in range(steps):
        a, b = one_step()
        t_fit += a
        t_fold += b
    t_fit /= steps
    t_fold /= steps
    scale = P / n_folds
    t_fit *= row_scale
    t_fold *= row_scale
    step_s = t_fit + t_fold * scale
    sample = ("full size: every row, every fold" if not loo else
              f"full-size fit, first {n_folds} of {P} folds per step, fold time scaled by {scale:.1f}")
    if row_scale != 1.0:
        sample = f"first {N} of {int(N * row_scale)} rows (the full matrix does not fit the host), every fold, time scaled linearly by {row_scale:.0f}"
    value = P / step_s
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "steps_requested": args.steps, "warmup_requested": args.warmup,
        "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32" if cfg.get("f32") else "f64", "data": "synthetic",
        "config": config_dict(CONFIGS[args.config], world),
        "reference_step": "Partitioner + fit + all folds (training_XTX_XTY), host arrays in, host arrays out, copy=False "
                          "(benchmarks/benchmark.py:52-158); runs on rank 0's host cores only",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "blas_threads": blas, "kind": kind, "sample": sample,
                         "fit_s": t_fit, "folds_s": t_fold * scale, "fold_path_value": P / (t_fold * scale)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# native arm
# ---------------------------------------------------------------------------------------------------------------
class Ctx:
    pass


def alloc_outputs(ctx, n, K, M):
    t = ctx.torch
    return dict(XTX=t.empty((n, K, K), dtype=t.float64, device=ctx.dev), XTY=t.empty((n, K, M), dtype=t.float64, device=ctx.dev),
                stats=t.empty((n, 2, K + M), dtype=t.float64, device=ctx.dev), scal=t.empty((n, 2), dtype=t.float64, device=ctx.dev),
                status=t.empty((n,), dtype=t.int32, device=ctx.dev))


DUMP_LIMIT_BYTES = 60_000_000   # keeps a dump, .npy headers included, under 64 MB


def dump_outputs(dirname, outs, first, n, K):
    """Writes the results the timed step left in `outs` (n folds, CSR fold numbers first, first + 1, ...) as
    dirname/<name>.npy: the arrays CVMatrix.training_batch returns, in the step's float dtype (status as float64),
    plus `folds` and `rows`, the CSR fold numbers and the XTX / XTY rows written (float64).  Where the n folds exceed
    DUMP_LIMIT_BYTES, a fixed seeded sample of them is written, and where one fold alone does, a fixed seeded sample
    of the rows of its XTX and XTY.  A step of more folds than one output window holds (leave-one-out: 4096 folds
    per chunk) leaves only its last chunk in `outs`, so the sample is drawn from that chunk."""
    import torch

    M = outs["XTY"].shape[2]
    item = outs["XTX"].element_size()
    per_fold = item * (K * K + K * M + 2 * (K + M) + 3)
    rng = np.random.default_rng(0)
    folds = np.arange(n)
    if n * per_fold > DUMP_LIMIT_BYTES:
        folds = np.sort(rng.choice(n, max(1, DUMP_LIMIT_BYTES // per_fold), replace=False))
    rows = np.arange(K)
    if per_fold > DUMP_LIMIT_BYTES:
        rows = np.sort(rng.choice(K, DUMP_LIMIT_BYTES // (2 * item * (K + M)), replace=False))
    dev = outs["XTX"].device
    fi, ri = torch.from_numpy(folds).to(dev), torch.from_numpy(rows).to(dev)
    pick = lambda name: outs[name].index_select(0, fi).cpu().numpy()  # noqa: E731
    mats = {name: outs[name].index_select(0, fi).index_select(1, ri).cpu().numpy() for name in ("XTX", "XTY")}
    stats, scal = pick("stats"), pick("scal")
    arrays = dict(mats, X_mean=stats[:, 0:1, :K], X_std=stats[:, 1:2, :K], Y_mean=stats[:, 0:1, K:], Y_std=stats[:, 1:2, K:],
                  sum_w_train=scal[:, 0], nnz_train=scal[:, 1], status=pick("status").astype(np.float64),
                  folds=(folds + first).astype(np.float64), rows=rows.astype(np.float64))
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a))
    print(f"bench.py: wrote {dirname}: {folds.size} of the {n} folds {first}..{first + n - 1}, {rows.size} of {K} rows of XTX "
          f"and XTY", file=sys.stderr)


def time_fold_path(ctx, m, P, steps, warmup, sf=None, row_sharded=False, clocks=False):
    """Device-timed fold path over all P folds of m's CSR: max over ranks of the CUDA-event time per step."""
    from cvmatrix_b200 import _lib

    torch, lib, h = ctx.torch, m._lib, m._h
    K, M = m.K, m.M or 0
    f0, f1 = (0, P) if row_sharded else (ctx.rank * P // ctx.world, (ctx.rank + 1) * P // ctx.world)
    # LOO writes 2.04 MB per fold: keep the resident output window bounded (it is rewritten every chunk)
    chunk = min(max(f1 - f0, 1), 4096) if not row_sharded else P
    outs = alloc_outputs(ctx, chunk, K, M)
    vp = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    _lib.check(lib.cvmx_set_stream(h, C.c_void_p(ctx.stream.cuda_stream)), h)

    def step():
        if row_sharded:
            sf.training_batch(0, P, out=outs, row_sharded=True)
            return
        for c0 in range(f0, f1, chunk):
            c1 = min(f1, c0 + chunk)
            _lib.check(lib.cvmx_training_batch(h, c0, c1, 3, vp(outs["XTX"]), vp(outs["XTY"]), vp(outs["stats"]), vp(outs["scal"]),
                                               vp(outs["status"]), _lib.DEVICE), h)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    _lib.check(lib.cvmx_profile_enable(h, 1), h)
    launches0 = m.launch_count
    sampler = ClockSampler(ctx.local_rank) if (clocks and ctx.rank == 0) else None
    if sampler:
        sampler.start()
    ctx.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    profiled = os.environ.get("BENCH_CUDA_PROFILER", "0") != "0"   # ncu --profile-from-start off: only the timed steps are captured
    if profiled:
        torch.cuda.profiler.start()
    e0.record(ctx.stream)
    for _ in range(steps):
        step()
    e1.record(ctx.stream)
    torch.cuda.synchronize()
    if profiled:
        torch.cuda.profiler.stop()
    ctx.barrier()
    ms = e0.elapsed_time(e1)
    clk = sampler.stop() if sampler else None
    launches = m.launch_count - launches0
    prof_ms, prof_n = (C.c_double * 3)(), (C.c_int64 * 3)()
    _lib.check(lib.cvmx_profile_read(h, prof_ms, prof_n), h)
    _lib.check(lib.cvmx_profile_enable(h, 0), h)
    if ctx.world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=ctx.dev)
        ctx.dist.all_reduce(t, op=ctx.dist.ReduceOp.MAX)
        ms = float(t.item())
    return dict(ms_per_step=ms / steps, prof_ms=[v / steps for v in prof_ms], prof_n=[v / steps for v in prof_n],
                launches=int(launches), clocks=clk, outs=outs, fold_range=(f0, f1), chunk=chunk,
                last_chunk=f0 + (f1 - f0 - 1) // chunk * chunk)   # first fold of the chunk the last step left in outs


def roofline_of(cfg_name, cfg, world, rank_rows, rank_folds, timing, ms_per_step):
    """Roofline of the dominant kernel on THIS rank: rank_rows validation rows contracted and rank_folds results
    written per step (SURVEY.md 8(d): flops = 2 N_val K (K+M) per fold, bytes = 2 s K (K+M) per fold)."""
    K, M = cfg["K"], cfg["M"]
    flops = 2.0 * rank_rows * K * (K + M)
    nbytes = 2.0 * 8 * K * (K + M) * rank_folds
    gram_ms, gram_n = timing["prof_ms"][1], timing["prof_n"][1]
    peak_tf, peak_src = fp64_peak_tflops()
    peak_bw, bw_src = hbm_peak_gbs()
    t_flop, t_byte = flops / (peak_tf * 1e12), nbytes / (peak_bw * 1e9)
    if t_flop >= t_byte:
        ach = flops / (gram_ms * 1e-3) / 1e12 if gram_ms > 0 else None
        roof = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf if ach else None,
                "peak_source": peak_src + "; FP64 tensor pipe", "kernel": "k_gram<double>"}
        if ach:
            # flops the kernel actually issues: tiles on / above the diagonal only, diagonal tiles at 3/4 (DESIGN.md 5.1)
            TI, TJ = -(-K // 128), -(-(K + M) // 128)
            issued_tiles = sum((0.75 if bj == bi else 1.0) for bi in range(TI) for bj in range(bi, TJ))
            issued = 2.0 * rank_rows * 128 * 128 * issued_tiles
            roof["issued_flops_per_step"] = issued
            roof["issued_frac_of_peak"] = issued / (gram_ms * 1e-3) / 1e12 / peak_tf
            roof["note"] = ("achieved / frac use the FULL flop count 2 N_val K (K+M) of SURVEY.md 8(d); XTX is symmetric, so only "
                            "upper-triangular tiles are computed and frac can exceed 1 - issued_frac_of_peak is the DMMA pipe's own load")
    else:
        ach = nbytes / (gram_ms * 1e-3) / 1e9 if gram_ms > 0 else None
        roof = {"bound": "hbm", "achieved": ach, "peak": peak_bw, "unit": "GB/s", "frac": ach / peak_bw if ach else None,
                "peak_source": bw_src, "kernel": "k_loo_operands + k_loo_tiles<double>",
                "note": "algorithmic bytes = read the resident total + write the result per fold (SURVEY.md 8(d)); the totals stay "
                        "in registers, so what reaches DRAM is the write half: write_gbs is achieved / 2",
                "write_gbs": ach / 2 if ach else None}
    roof.update({"traffic": None, "kernel_ms_per_step": gram_ms, "kernel_launches_per_step": gram_n,
                 "stats_ms_per_step": timing["prof_ms"][0], "reduce_ms_per_step": timing["prof_ms"][2],
                 "algorithmic_flops_per_step": flops, "algorithmic_bytes_per_step": nbytes, "per": "rank 0" if world > 1 else "GPU",
                 "step_roofline_frac": max(t_flop, t_byte) / (ms_per_step * 1e-3)})
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        shards = int(os.environ.get("BENCH_EMULATE_SHARDS", "0")) or world
        roof["traffic"] = tj.get(cfg_name if shards == 1 else f"{cfg_name}@{shards}")   # ncu capture of the same per-rank launch
    except Exception:
        pass
    return roof


def run_row_slabs(args, cfg, ctx):
    """BASELINE config 5 at full size: N = 2M x K = 5000 (82 GB float64) is produced block by block ON THE DEVICE (it
    cannot exist on the host) and its ROWS are sharded across the ranks (cvmatrix_b200.distributed.RowSlabFolds)."""
    from cvmatrix_b200 import CVMatrix, _lib, sharding
    from cvmatrix_b200.distributed import RowSlabFolds

    torch, dist, dev, rank, world = ctx.torch, ctx.dist, ctx.dev, ctx.rank, ctx.world
    N, K, M, P = cfg["N"], cfg["K"], cfg["M"], cfg["P"]
    f32 = bool(cfg.get("f32"))
    npdt, tdt = (np.float32, torch.float32) if f32 else (np.float64, torch.float64)
    B = 65536
    steps = args.steps
    warmup = 1

    gw = torch.Generator(device=dev)
    gw.manual_seed(4242)
    w = torch.rand((N,), dtype=torch.float64, generator=gw, device=dev).to(tdt)      # the same on every rank
    r0, r1 = sharding.slab_rows(rank, world, N)

    def blocks():
        for blk in range(r0 // B, (r1 + B - 1) // B):
            g = torch.Generator(device=dev)
            g.manual_seed(42_000 + blk)                                              # block-seeded: independent of the world size
            full = torch.rand((min(N, (blk + 1) * B) - blk * B, K + M), dtype=torch.float64, generator=g, device=dev).to(tdt)
            lo, hi = max(r0, blk * B), min(r1, (blk + 1) * B)
            part = full[lo - blk * B: hi - blk * B]
            torch.cuda.current_stream(dev).synchronize()                             # the library reads the block on ITS stream
            yield lo, part[:, :K], part[:, K:]

    m = CVMatrix(dtype=npdt, device=ctx.local_rank)
    lib, h = m._lib, m._h
    rs = RowSlabFolds(m, N, K, M, w, block_rows=B)
    # generation is not part of fit: measure it alone first (the same kernels, results dropped)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in blocks():
        pass
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    ctx.barrier()
    t0 = time.perf_counter()
    rs.fit(blocks())
    torch.cuda.synchronize()
    ctx.barrier()
    fit_s = time.perf_counter() - t0 - gen_s
    torch.cuda.empty_cache()
    folds = np.arange(N) % P
    order = np.argsort(folds, kind="stable")
    offsets = np.concatenate([[0], np.cumsum(np.bincount(folds, minlength=P))]).astype(np.int64)
    rs.set_folds((offsets, order))
    o0, o1 = sharding.fold_block(rank, world, 0, P)
    outs = rs.alloc_outputs(max(o1 - o0, 1))
    _lib.check(lib.cvmx_set_stream(h, C.c_void_p(ctx.stream.cuda_stream)), h)

    def step():
        rs.training_batch(0, P, out=outs)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    _lib.check(lib.cvmx_profile_enable(h, 1), h)
    launches0 = m.launch_count
    sampler = ClockSampler(ctx.local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ctx.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    profiled = os.environ.get("BENCH_CUDA_PROFILER", "0") != "0"   # ncu --profile-from-start off: only the timed steps are captured
    if profiled:
        torch.cuda.profiler.start()
    e0.record(ctx.stream)
    for _ in range(steps):
        step()
    e1.record(ctx.stream)
    torch.cuda.synchronize()
    if profiled:
        torch.cuda.profiler.stop()
    ctx.barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    launches = m.launch_count - launches0
    prof_ms, prof_n = (C.c_double * 3)(), (C.c_int64 * 3)()
    _lib.check(lib.cvmx_profile_read(h, prof_ms, prof_n), h)
    _lib.check(lib.cvmx_profile_enable(h, 0), h)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs, o0, o1 - o0, K)
    # end to end: fit from the device-generated blocks + all folds + every result copied to pinned host memory
    host_out = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in outs.items() if v is not None}
    ctx.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rs.fit(blocks())
    rs.set_folds((offsets, order))
    res = rs.training_batch(0, P, out=outs)
    n_own = res["fold_end"] - res["fold_begin"]
    d2h = 0
    for k, hb in host_out.items():
        if n_own > 0:
            hb[:n_own].copy_(outs[k][:n_own], non_blocking=True)
            d2h += hb[:n_own].numel() * hb.element_size()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0 - gen_s
    if world > 1:
        t = torch.tensor([ms, fit_s, e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, fit_s, e2e_s = (float(v) for v in t.tolist())
        t = torch.tensor([float(d2h)], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        d2h = int(t.item())
    ms_per_step = ms / steps
    if rank != 0:
        return
    flops = 2.0 * (r1 - r0) * K * (K + M)                    # this rank's rows, every one in exactly one fold
    gram_ms = prof_ms[1] / steps
    peak_tf, peak_src = fp64_peak_tflops()
    ach = flops / (gram_ms * 1e-3) / 1e12 if gram_ms > 0 else None
    TI, TJ = -(-K // 128), -(-(K + M) // 128)
    issued = 2.0 * (r1 - r0) * 128 * 128 * sum((0.75 if bj == bi else 1.0) for bi in range(TI) for bj in range(bi, TJ))
    roof = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf if ach else None,
            "peak_source": peak_src + "; FP64 tensor pipe" + (" (float32 data, float64 DMMA accumulation)" if f32 else ""),
            "kernel": "k_gram<%s>" % ("float" if f32 else "double"), "issued_flops_per_step": issued,
            "issued_frac_of_peak": issued / (gram_ms * 1e-3) / 1e12 / peak_tf if gram_ms > 0 else None,
            "note": "achieved / frac use the FULL flop count 2 N K (K+M) of SURVEY.md 8(d) for this rank's rows; only upper-triangular tiles are issued",
            "traffic": None, "kernel_ms_per_step": gram_ms, "kernel_launches_per_step": prof_n[1] / steps,
            "stats_ms_per_step": prof_ms[0] / steps, "reduce_ms_per_step": prof_ms[2] / steps,
            "algorithmic_flops_per_step": flops, "per": "rank 0" if world > 1 else "GPU",
            "step_roofline_frac": flops / (peak_tf * 1e12) / (ms_per_step * 1e-3)}
    line = {
        "metric": METRIC, "value": P / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "steps_requested": args.steps, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32" if f32 else "f64", "data": "synthetic (uniform [0,1), generated block by block on the device, block-seeded)",
        "config": config_dict(cfg, world),
        "collective": ("peer-memory reduction over NVLink (symmetric memory, no all-reduce)" if rs._symm is not None else
                       ("1 NCCL all-reduce of the fold Grams" if world > 1 else None)),
        "clocks": clocks,
        "e2e": {"value": P / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(offsets.nbytes + order.nbytes), "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_s * 1e3, "steps": 1,
                "includes": "fit streamed from device-generated row blocks (the 80 GB matrix cannot exist on the host; generation time "
                            "subtracted) + chained sums + totals all-reduce + set_folds + all folds + D2H of every output into pinned memory"},
        "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": None,
        "parity": {"note": "no host can hold this matrix: parity of this path is pinned at reduced N - tests/test_gpu_fullsize.py::"
                           "test_cfg5_reduced_wide_k (K = 5000, one GPU) and the row-slab section of tests/dist_fit_worker.py (2 GPUs) against the oracle"},
        "fit_s": fit_s, "generation_s": gen_s, "resident_gb_per_gpu": (r1 - r0) * (-(-(K + M) // 32) * 32) * (4 if f32 else 8) / 1e9,
    }
    print(json.dumps(line), flush=True)


def native_fold_results(m, folds_idx, K):
    """Host copies of the batched path's results for the given CSR fold numbers (XTX, XTY, 4 statistics rows)."""
    res = {}
    for f in folds_idx:
        r = m.training_batch(f, f + 1, out="numpy")
        res[f] = (r["XTX"][0], r["XTY"][0], (r["X_mean"][0], r["X_std"][0], r["Y_mean"][0], r["Y_std"][0]))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the cfg3 / cfg4 lines appended to the default (cfg2) run")
    ap.add_argument("--no-parity", action="store_true", help="skip the comparison with the CPU reference (N > 1: one fold on rank 0)")
    ap.add_argument("--e2e-out", default="numpy", choices=["numpy", "pinned"],
                    help="host destination of the e2e results: fresh numpy arrays (the reference's convention) or the reused page-locked pool")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (above 64 MB, or beyond one output window of "
                         "4096 folds: a fixed, seeded sample of the last window)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.dump_outputs and (args.impl != "native" or world > 1 or os.environ.get("BENCH_EMULATE_SHARDS", "0") != "0"):
        ap.error("--dump-outputs writes the native path's results of a single process (--impl native, one rank, no shard emulation)")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup

    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    import torch
    import torch.distributed as dist

    from cvmatrix_b200 import CVMatrix, Partitioner, _lib, sharding
    from cvmatrix_b200.distributed import ShardedFolds, fit_sharded_upload

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries ONE JSON line: NCCL's own log (NCCL_DEBUG=INFO / VERSION, from the environment or nccl.conf) is
        # NOT silenced - it goes to stderr unless the caller already pointed it at a file
        if not os.environ.get("NCCL_DEBUG_FILE"):
            os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        dist.init_process_group("nccl", device_id=dev)

    ctx = Ctx()
    ctx.torch, ctx.dist, ctx.dev, ctx.rank, ctx.world, ctx.local_rank = torch, dist, dev, rank, world, local_rank
    ctx.barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)
    ctx.stream = torch.cuda.Stream(dev)   # a real (non-default) stream shared by the library and the timing events
    torch.cuda.set_stream(ctx.stream)

    if cfg.get("device_generated"):
        run_row_slabs(args, cfg, ctx)
        if world > 1:
            dist.destroy_process_group()
        return

    N, K, M, P = cfg["N"], cfg["K"], cfg["M"], cfg["P"]
    X, Y, w, folds, keep = make_host_inputs(cfg, pinned=True)
    part = Partitioner(folds)
    m = CVMatrix(dtype=np.float64, copy=False, device=local_rank)
    lib, h = m._lib, m._h
    t0 = time.perf_counter()
    m.fit(X, Y, w)
    fit_upload_s = time.perf_counter() - t0
    m.set_folds(part)

    row_sharded = sharding.use_row_sharding(P, world)
    assert row_sharded == row_sharded_mode(P, world)
    sf = ShardedFolds(m) if world > 1 else None
    emulate = int(os.environ.get("BENCH_EMULATE_SHARDS", "0"))   # profiling aid: rank 0's share of an N-way sharded step
    if emulate and world == 1:
        sf = ShardedFolds(m)
        sf.emulate_shards = emulate
        row_sharded = True

    # ---- the timed region: fold path, inputs resident -------------------------------------------------------
    tm = time_fold_path(ctx, m, P, args.steps, args.warmup, sf=sf, row_sharded=row_sharded, clocks=True)
    ms_per_step = tm["ms_per_step"]
    value = P / (ms_per_step * 1e-3)
    f0, f1 = tm["fold_range"]
    shards = emulate or world
    if row_sharded:
        rank_rows, rank_folds = int(part.offsets[P]) // shards, P / shards
    else:
        rank_rows, rank_folds = int(part.offsets[f1] - part.offsets[f0]), f1 - f0
    roof = roofline_of(args.config, cfg, world, rank_rows, rank_folds, tm, ms_per_step)
    outs, clocks, launches = tm["outs"], tm["clocks"], tm["launches"]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs, tm["last_chunk"], f1 - tm["last_chunk"], K)

    # results of the timed path for the parity block (before e2e refits the handle)
    want_parity = not args.no_parity and not emulate
    native_res, owner_of = {}, {}
    if want_parity:
        if world == 1:
            if not args.no_cpu_baseline:
                native_res = native_fold_results(m, list(range(min(P, 5))) if P <= 1000 else [0, 1, P // 2, P - 1], K)
        elif row_sharded:
            # fold 0 of the row-sharded step, fetched from its owner (rank 0 may own no fold)
            o = [sharding.fold_block(r, world, 0, P) for r in range(world)]
            src = next(r for r, (a, b) in enumerate(o) if a <= 0 < b)
            torch.cuda.synchronize()
            bufs = [outs["XTX"][:1].clone(), outs["XTY"][:1].clone(), outs["stats"][:1].clone()]   # owner: its fold 0 sits first
            for b in bufs:
                dist.broadcast(b, src=src)
            if rank == 0:
                st = bufs[2][0].cpu().numpy()
                native_res[0] = (bufs[0][0].cpu().numpy(), bufs[1][0].cpu().numpy(), (st[0, :K], st[1, :K], st[0, K:], st[1, K:]))
        else:
            torch.cuda.synchronize()
            if rank == 0:     # first fold of rank 0's own block
                lo = tm["last_chunk"]   # the chunk that is still in the output window
                st = outs["stats"][0].cpu().numpy()
                native_res[lo] = (outs["XTX"][0].cpu().numpy(), outs["XTY"][0].cpu().numpy(), (st[0, :K], st[1, :K], st[0, K:], st[1, K:]))

    # ---- the other single-box workloads, device-timed in the same process (default run only) -----------------
    also = None
    if args.config == "cfg2" and not args.no_also and not emulate:
        also = {}
        a_steps, a_warm = args.steps, args.warmup
        c3 = CONFIGS["cfg3"]
        m.set_folds(Partitioner(np.arange(N) % c3["P"]))
        t3 = time_fold_path(ctx, m, c3["P"], a_steps, a_warm)
        b3 = (rank * c3["P"] // world, (rank + 1) * c3["P"] // world)
        also["cfg3"] = {"workload": c3["name"], "value": c3["P"] / (t3["ms_per_step"] * 1e-3), "unit": UNIT, "ms_per_step": t3["ms_per_step"],
                        "steps": a_steps, "warmup": a_warm, "n_gpus": world, "parallelism": f"fold-sharded x{world}", "gpu_launches": t3["launches"],
                        "roofline": roofline_of("cfg3", c3, world, (b3[1] - b3[0]) * (N // c3["P"]), b3[1] - b3[0], t3, t3["ms_per_step"])}
        del t3
        c4 = CONFIGS["cfg4"]
        X4, Y4, w4, folds4, keep4 = make_host_inputs(c4, pinned=False)
        m4 = CVMatrix(dtype=np.float64, copy=False, device=local_rank)
        m4.fit(X4, Y4, w4)
        m4.set_folds(Partitioner(folds4))
        t4 = time_fold_path(ctx, m4, c4["P"], a_steps, a_warm)
        b4 = (rank * c4["P"] // world, (rank + 1) * c4["P"] // world)
        also["cfg4"] = {"workload": c4["name"], "value": c4["P"] / (t4["ms_per_step"] * 1e-3), "unit": UNIT, "ms_per_step": t4["ms_per_step"],
                        "steps": a_steps, "warmup": a_warm, "n_gpus": world, "parallelism": f"fold-sharded x{world}", "gpu_launches": t4["launches"],
                        "roofline": roofline_of("cfg4", c4, world, b4[1] - b4[0], b4[1] - b4[0], t4, t4["ms_per_step"])}
        _lib.check(m4._lib.cvmx_set_stream(m4._h, None), m4._h)
        del t4, m4, X4, Y4, w4
        torch.cuda.empty_cache()
        m.set_folds(part)
    del tm

    # ---- end to end through the public API, host buffers in, host arrays out ------------------------------
    e2e = None
    e2e_res = {}
    if not args.no_e2e:
        if world == 1:
            _lib.check(lib.cvmx_set_stream(h, None), h)
        e2e_steps = args.steps
        out_bytes = 0
        host_out = None
        fb0, fb1 = rank * P // world, (rank + 1) * P // world
        chunk = min(max(fb1 - fb0, 1), 4096)
        if row_sharded and world > 1:   # pinned host buffers for the folds this rank owns
            o0, o1 = sharding.fold_block(rank, world, 0, P)
            n_own = max(o1 - o0, 1)
            host_out = {k: torch.empty((n_own,) + tuple(outs[k].shape[1:]), dtype=outs[k].dtype, pin_memory=True)
                        for k in ("XTX", "XTY", "stats", "scal", "status")}

        parts = {"partitioner_ms": 0.0, "fit_ms": 0.0, "set_folds_ms": 0.0, "folds_ms": 0.0}

        # several GPUs, few huge folds: the e2e path keeps the ROWS sharded (row slabs): every rank uploads only its own
        # 1 / world of the rows over its PCIe link and nothing is exchanged but the chained column sums (2 ld values per
        # hop) and the per-slab Grams the fold owners sum over NVLink
        slab = None
        if row_sharded and world > 1:
            from cvmatrix_b200.distributed import RowSlabFolds, upload_balanced_bounds

            # slab sizes follow the copy rate each rank reaches while all ranks upload at once (set-up, outside the timed region)
            bounds = None
            if os.environ.get("BENCH_BALANCED_SLABS", "1") != "0":
                n_s = min(N // world, max(8192, (128 << 20) // (8 * K)))
                bounds = upload_balanced_bounds(N, keep[0][rank * (N // world): rank * (N // world) + n_s], dev)
            slab = RowSlabFolds(m, N, K, M, w, block_rows=32768, bounds=bounds)
            w_pinned = torch.from_numpy(w)

        def e2e_step(Xh, Yh, wh, keep_results=False):
            nonlocal out_bytes
            t0 = time.perf_counter()
            p2 = Partitioner(folds)
            t1 = time.perf_counter()
            if slab is not None:
                slab.w.copy_(w_pinned, non_blocking=True)                      # the weights are inputs too (8 MB)
                r0, r1 = slab.row0, slab.row1
                slab.fit((b0, Xh[b0:min(r1, b0 + 32768)], Yh[b0:min(r1, b0 + 32768)]) for b0 in range(r0, r1, 32768))
                t2 = time.perf_counter()
                slab.set_folds(p2)
            elif world > 1:
                # every rank uploads 1 / world of the rows over its own PCIe link; slabs are exchanged over NVLink
                fit_sharded_upload(m, Xh, Yh, wh)
                t2 = time.perf_counter()
                m.set_folds(p2)
            else:
                # fit + set_folds in one call: the folds partition the rows, so every row is contracted once, per fold,
                # behind the upload (XtWX = sum of the fold Grams) and training_batch only finishes the folds
                m.fit(Xh, Yh, wh, folds=p2)
                t2 = time.perf_counter()
            t3 = time.perf_counter()
            out_bytes = 0
            if row_sharded and world > 1:
                res = slab.training_batch(0, P, out=outs)
                n = res["fold_end"] - res["fold_begin"]
                for k, hbuf in host_out.items():
                    if n > 0:
                        hbuf[:n].copy_(outs[k][:n], non_blocking=True)
                        out_bytes += hbuf[:n].numel() * hbuf.element_size()
                torch.cuda.synchronize()
            else:
                for c0 in range(fb0, fb1, chunk):
                    r = m.training_batch(c0, min(fb1, c0 + chunk), out=args.e2e_out)
                    out_bytes += r["XTX"].nbytes + r["XTY"].nbytes + 2 * r["X_mean"].nbytes + 2 * r["Y_mean"].nbytes
                    if keep_results and c0 == fb0 and P <= 1000:
                        for f in range(min(P, 5)):
                            e2e_res[f] = (r["XTX"][f].copy(), r["XTY"][f].copy(),
                                          (r["X_mean"][f].copy(), r["X_std"][f].copy(), r["Y_mean"][f].copy(), r["Y_std"][f].copy()))
            t4 = time.perf_counter()
            for k, v in zip(parts, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
                parts[k] += v * 1e3

        if world > 1:
            _lib.check(lib.cvmx_set_stream(h, C.c_void_p(ctx.stream.cuda_stream)), h)
        e2e_step(X, Y, w)
        for k in parts:
            parts[k] = 0.0
        ctx.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            e2e_step(X, Y, w, keep_results=(i == e2e_steps - 1 and world == 1 and want_parity and not args.no_cpu_baseline))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        h2d = int(X.nbytes + Y.nbytes + w.nbytes) // world + int(part.indices.nbytes + part.offsets.nbytes)
        if world > 1:
            t = torch.tensor([dt, float(out_bytes)], dtype=torch.float64, device=dev)
            dist.all_reduce(t[:1], op=dist.ReduceOp.MAX)
            dist.all_reduce(t[1:], op=dist.ReduceOp.SUM)
            dt, out_bytes = float(t[0].item()), int(t[1].item())
            h2d *= world
        e2e = {"value": P / (dt / e2e_steps), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": int(out_bytes), "ms_per_step": dt / e2e_steps * 1e3, "steps": e2e_steps,
               "includes": ("Partitioner + fit (H2D from pinned host memory" + ((f": a slab of the rows per rank (sizes proportional to the measured copy rates: {[b - a for a, b in zip(bounds, bounds[1:])] if bounds else 'equal'}), rows stay sharded (row slabs: chained column sums, per-slab Grams summed by the fold owners over NVLink)" if slab is not None else f": 1/{world} of the rows per rank, slabs exchanged over NVLink") if world > 1 else "; fused with the fold Grams when the folds partition the rows")
                            + ") + set_folds + all folds + D2H of every output"),
               "host_outputs": args.e2e_out, "breakdown_ms": {k: v / e2e_steps for k, v in parts.items()}}
        if world == 1 and N * K * 8 <= 5e9 and P <= 1000:
            # the same call with ordinary (pageable) numpy arrays, as a drop-in user would pass them
            Xp, Yp, wp = np.array(X), np.array(Y), np.array(w)
            e2e_step(Xp, Yp, wp)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                e2e_step(Xp, Yp, wp)
            torch.cuda.synchronize()
            dtp = (time.perf_counter() - t0) / args.steps
            e2e["pageable_input"] = {"value": P / dtp, "unit": UNIT, "ms_per_step": dtp * 1e3, "steps": args.steps,
                                     "note": "inputs are ordinary (pageable) numpy arrays: the library stages them through its page-locked ring filled by worker threads "
                                             "(csrc/host_stager.h; CVMX_HOST_STAGER=0 = the driver's bounce buffer, ~370 ms)"}
            del Xp, Yp, wp

    # ---- CPU baseline + parity: the reference on this box's host cores (rank 0) --------------------------------
    cpu = parity = parity_e2e = None
    if rank == 0 and ((world == 1 and not args.no_cpu_baseline) or (world > 1 and want_parity and native_res)):
        RefCV, RefPart, kind, threads, blas = load_reference()
        t0 = time.perf_counter()
        op = RefPart(folds)
        orc = RefCV(dtype=np.float64, copy=False)
        orc.fit(X, Y, w)
        t_fit = time.perf_counter() - t0
        keys = list(op.folds_dict)
        if world == 1:
            n_f = len(keys) if P <= 5 else max(5, min(len(keys), int(12.0 / (9.0 / P if P <= 1000 else 0.005))))
            n_f = min(n_f, 2000)
            timed = keys[:n_f]
        else:
            timed = [keys[f] for f in sorted(native_res)]
            n_f = len(timed)
        ref_res = {}
        pos_of = {k: i for i, k in enumerate(keys)}
        needed = set(native_res) | set(e2e_res)
        t0 = time.perf_counter()
        for k in timed:
            (rx, ry), rs = orc.training_XTX_XTY(op.get_validation_indices(k))
            if pos_of[k] in needed:
                ref_res[pos_of[k]] = (rx, ry, rs)
        t_folds = (time.perf_counter() - t0) * (len(keys) / n_f)
        for pos in native_res:
            if pos not in ref_res:     # folds outside the timed sample (leave-one-out: the sample is a prefix)
                (rx, ry), rs = orc.training_XTX_XTY(op.get_validation_indices(keys[pos]))
                ref_res[pos] = (rx, ry, rs)
        if world == 1:
            cpu = {"value": P / t_folds, "unit": UNIT, "cores": threads, "blas_threads": blas, "kind": kind,
                   "sample": f"full-size fit ({t_fit:.1f} s, not in value) then {n_f} of {P} folds, fold-path time scaled to {P} folds",
                   "fit_s": t_fit, "folds_s": t_folds, "e2e_value": P / (t_fit + t_folds)}
        if want_parity:
            what = ("timed path: plain fit + batched fold path" if world == 1 else
                    f"timed path on {world} GPUs, fold {sorted(native_res)[0]} as returned by its owner")
            parity = parity_summary([parity_entry(native_res[p], ref_res[p]) for p in sorted(native_res)], kind, what)
            if e2e_res:
                parity_e2e = parity_summary([parity_entry(e2e_res[p], ref_res[p]) for p in sorted(e2e_res) if p in ref_res], kind,
                                            "e2e path: fit(folds=...) fused with the fold Grams, results as copied to the host")
        del orc
    ctx.barrier()

    if rank == 0:
        collective = None
        if row_sharded and world > 1:
            collective = ("peer-memory reduction over NVLink (symmetric memory, no all-reduce)" if (sf is not None and sf._symm is not None)
                          else "1 NCCL all-reduce")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config_dict(cfg, world), "collective": collective, "clocks": clocks,
            "e2e": e2e, "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu, "parity": parity,
            "parity_e2e_path": parity_e2e, "also": also, "fit_with_h2d_s": fit_upload_s,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
