#!/usr/bin/env python
"""
bench.py -- GP posteriors/s at N=16384 (BASELINE.json metric) on N GPUs of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  (N > 1: launched by torchrun, one rank per GPU; ranks process independent posterior draws -- the
   path's natural sharding, SURVEY.md section 8e "draw-parallel" -- so scaling is weak and there is no
   data-path collective; torch.distributed is used only for the barrier and the max-over-ranks.)

A "step" is one pass of the hot path over one batch of S hyper-parameter draws: for each draw
Gram(k_XX) -> N x N Cholesky -> Gram(k_pX) -> triangular solves -> posterior mean + diagonal variance
(the replacement of gpax/models/gp.py:253-277 under the vmap of gp.py:393-395).

  value   posteriors/s with X, y, X_new, theta resident in HBM (device-pointer C-ABI call)
  e2e     the same through the host-buffer C-ABI call (pinned host memory in, host memory out:
          H2D of X, y, X_new, theta and D2H of mean, var, info inside the timed region)
  roofline  dominant kernel = the trailing-update SYRK of the N=16384 factorisation (8192 x 8192, k = 8192, lower half),
          which runs on the int8 tcgen05 tensor cores (oz_mma_kernel, 6 base-256 digit planes = 21 exact int8 GEMMs): achieved int8
          TOP/s from its CUDA-event duration against 2 x the measured bf16 peak of MEASURED_PEAKS.json; the fp64-equivalent
          rate and its ratio to the cuBLAS DGEMM rate measured live are reported beside it, and `roofline_dmma` gives the
          fp64 DMMA kernel on the same launch
  cpu_baseline  the oracle's restatement of the reference formulation (explicit inverse,
          oracle.exact_posterior) timed on the host cores on a bounded sample

--dump-outputs DIR writes what the last timed step returned, mean.npy and var.npy ([S, P] float64), so that two builds
can be compared output for output: the inputs depend only on the seed, the rank and --draws.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1 to every rank.  Rank 0 also times the CPU baseline / the reference arm, which are
# to use all host cores, and OpenBLAS fixes its pool when NumPy is imported: lift the cap on rank 0 before that import.
if os.environ.get("RANK", "0") == "0" and os.environ.get("OMP_NUM_THREADS") == "1" and "TORCHELASTIC_RUN_ID" in os.environ:
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count())
    os.environ["OPENBLAS_NUM_THREADS"] = str(os.cpu_count())

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HOST_MS = []
WORKLOAD = dict(name="exactgp_rbf_N16384_d3_P1024", N=16384, d=3, P=1024, kernel="RBF", ell=0.3, scale=1.0, noise=0.1,
                jitter=1e-6, S=8)


def make_inputs(rank):
    """SURVEY.md section 8d 'headline' row: N=16384, d=3, U(0,1)^3, seed 4 (+rank), RBF l=0.3, noise 0.1, P=1024."""
    w = WORKLOAD
    rng = np.random.default_rng(4 + 1000 * rank)
    X = rng.uniform(0, 1, (w["N"], w["d"]))
    y = np.sin(3 * X[:, 0]) * np.cos(2 * X[:, 1]) + X[:, 2] + 0.1 * rng.standard_normal(w["N"])
    Xn = rng.uniform(0, 1, (w["P"], w["d"]))
    # S draws around the nominal hyper-parameters (every draw is a different K: nothing can be cached)
    S = w["S"]
    theta = np.empty((S, w["d"] + 3))
    theta[:, :w["d"]] = w["ell"] * np.exp(0.05 * rng.standard_normal((S, w["d"])))
    theta[:, w["d"]] = w["scale"] * np.exp(0.05 * rng.standard_normal(S))
    theta[:, w["d"] + 1] = w["noise"] * np.exp(0.05 * rng.standard_normal(S))
    theta[:, w["d"] + 2] = 1.0
    return X, y, Xn, theta


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:  # noqa: BLE001
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# stdout carries exactly ONE line, the JSON result: libraries that write to the C-level stdout (NCCL prints its version
# banner there) are diverted to stderr for the life of the process and the result goes to the saved descriptor.
_RESULT_FD = os.dup(1)
os.dup2(2, 1)


def emit(text):
    sys.stdout.flush()
    os.write(_RESULT_FD, (text + "\n").encode())


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    td = None
    if world > 1:
        import torch
        import torch.distributed as td_
        torch.cuda.set_device(local)
        td_.init_process_group("nccl", device_id=torch.device("cuda", local))
        td = td_
    return rank, world, local, td


def barrier_sync(td, local):
    if td is not None:
        import torch
        td.barrier()
        torch.cuda.synchronize(local)


def max_over_ranks(td, local, value):
    if td is None:
        return value
    import torch
    t = torch.tensor([value], dtype=torch.float64, device=f"cuda:{local}")
    td.all_reduce(t, op=td.ReduceOp.MAX)
    return float(t.item())


def measure_fp64_peak(local):
    """cuBLAS DGEMM 8192^3 (torch.matmul fp64), best of 5 after warm-up, CUDA events: the fp64 denominator."""
    import torch
    dev = f"cuda:{local}"
    a = torch.randn(8192, 8192, dtype=torch.float64, device=dev)
    b = torch.randn(8192, 8192, dtype=torch.float64, device=dev)
    for _ in range(2):
        a @ b
    torch.cuda.synchronize(dev)
    best = 1e30
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        a @ b
        e1.record()
        torch.cuda.synchronize(dev)
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2 * 8192 ** 3 / best / 1e9  # TFLOP/s


def measure_dominant_kernel(ctx, ffi):
    """The trailing-update SYRK at the headline size (8192 x 8192, k = 8192, lower half), device resident, CUDA events
    around the launch(es), through the int8 tcgen05 path (default) and through the fp64 DMMA path."""
    n = 8192
    rng = np.random.default_rng(0)
    A = ctx.to_device(rng.standard_normal((n, n)))
    Cm = ctx.to_device(np.zeros((n, n)))
    out = {}
    w = WORKLOAD
    # the plane count the library's accuracy rule picks for this workload (oz_auto_planes in common.cuh)
    planes = 6 if (w["N"] * w["scale"] + w["noise"] + w["jitter"]) / (w["noise"] + w["jitter"]) <= 1e6 else 7
    for name, oz in (("dmma", 0), ("tcgen05_i8", planes)):
        ctx.set_option("ozaki", oz)
        ms = []
        for _ in range(5):
            ctx._check(ctx.lib.b2gp_gemm_nt(ctx.h, n, n, n, -1.0, A.ptr, n, A.ptr, n, 1.0, Cm.ptr, n, 1, ffi.FLAG_DEVICE_PTRS))
            ms.append(ctx.last_timing()["epilogue_ms"])
        ms = float(np.mean(ms[2:]))
        out[name] = {"ms": ms, "fp64_equiv_tflops": float(n) ** 3 / ms / 1e9}
    ctx.set_option("ozaki", -1)
    A.free()
    Cm.free()
    out["planes"] = planes
    out["pairs"] = planes * (planes + 1) // 2
    out["int8_ops_per_launch"] = out["pairs"] * float(n) ** 3          # 2 * (n*n/2) * n MACs per digit-plane pair
    return out


def cpu_baseline(budget_s=30.0):
    """The oracle on the host cores, bounded samples.  `value` is the reference formulation (explicit inverse, 2 N^3:
    what gpax's own CPU path does); `best_cpu_formulation` is the same posterior by Cholesky (N^3 / 3), reported so
    that the GPU/CPU ratio is not inflated by the reference's choice of algorithm (SURVEY 8d)."""
    import oracle
    w = WORKLOAD
    cores = os.cpu_count()
    rng = np.random.default_rng(4)
    params = {"k_length": np.full(w["d"], w["ell"]), "k_scale": w["scale"], "noise": w["noise"]}

    def run(N, fn):
        X = rng.uniform(0, 1, (N, w["d"]))
        y = rng.standard_normal(N)
        Xn = rng.uniform(0, 1, (w["P"], w["d"]))
        t0 = time.perf_counter()
        fn(X, y, Xn, params, "RBF", jitter=w["jitter"])
        return time.perf_counter() - t0

    def sample(fn, what, budget):
        """one posterior at the largest N <= 16384 that fits the budget, scaled to N = 16384 with the growth factor per
        doubling MEASURED on this host between the last two sizes (a 128-core LAPACK run grows by ~3.8x per doubling here,
        not by the 8x of the flop count: the `--impl reference` arm, which times N = 16384 itself, is the check)"""
        run(1024, fn)
        times = {2048: run(2048, fn), 4096: run(4096, fn)}
        N = 4096
        while N * 2 <= w["N"] and times[N] * (times[N] / times[N // 2]) <= budget:
            N *= 2
            times[N] = run(N, fn)
        if N == w["N"]:
            return {"value": 1.0 / times[N], "sample": f"1 posterior at N={N} P={w['P']} ({what}), {times[N]:.1f} s, no scaling"}
        growth = times[N] / times[N // 2]
        scaled = times[N] * growth ** int(round(np.log2(w["N"] / N)))
        return {"value": 1.0 / scaled, "sample": f"1 posterior at N={N} ({times[N]:.1f} s, {what}) scaled to N={w['N']} by the measured growth per "
                                                   f"doubling ({growth:.2f}x from N={N // 2} to N={N}) = {scaled:.1f} s"}

    ref = sample(oracle.exact_posterior, "oracle.exact_posterior, explicit inverse as gp.py:271", budget_s)
    best = sample(oracle.exact_posterior_chol, "oracle.exact_posterior_chol, scipy cho_factor / cho_solve", budget_s / 2)
    return {"value": ref["value"], "unit": "posteriors/s", "cores": cores, "kind": "port", "sample": ref["sample"],
            "best_cpu_formulation": {"value": best["value"], "unit": "posteriors/s", "sample": best["sample"]}}


DUMP_LIMIT_BYTES = 63 * 10 ** 6        # 64 MB less room for the .npy headers


def dump_outputs(out_dir, arrays, suffix=""):
    """Write each [S, P] array as out_dir/<name><suffix>.npy.  Above DUMP_LIMIT_BYTES in all, the same seeded sample of
    draws (rows) is kept from every array and its row indices go to draws<suffix>.npy."""
    os.makedirs(out_dir, exist_ok=True)
    S = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a[0].nbytes for a in arrays.values()) + 8          # + the row's index in draws.npy
    keep = min(S, DUMP_LIMIT_BYTES // row_bytes)
    if keep < S:
        rows = np.sort(np.random.default_rng(0).choice(S, keep, replace=False))
        arrays = dict({k: a[rows] for k, a in arrays.items()}, draws=rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def dist_workloads(ctx, ffi, rank, world, local, td, steps=3):
    """The two BASELINE configs whose data path has a real exchange step (SURVEY.md section 8e), run inside libb200gp.so over
    NCCL (gpax_b200/csrc/dist.cuh) -- STRONG scaling, reported as extra objects of the bench line:
      c4  ExactGP RBF N=32768 d=3 P=1024: k_XX 2-D block-cyclic over the process grid (2 x 4 on 8 GPUs), panel broadcast /
          all-gather on row / column communicators, one posterior (mean + diag variance) per step
      c5  viSparseGP Matern N=262144 d=2, M=4096 inducing points, P=4096: N-sharded statistics + one M x M all-reduce
    With one GPU the same problems run through the single-GPU entry points (the strong-scaling baseline)."""
    from gpax_b200 import dist
    out = {}
    # ---- c4
    N, d, P, nb = 32768, 3, 1024, 512
    rng = np.random.default_rng(5)
    X = rng.uniform(0, 1, (N, d))
    y = np.sin(3 * X[:, 0]) * np.cos(2 * X[:, 1]) + X[:, 2] + 0.1 * rng.standard_normal(N)
    Xn = rng.uniform(0, 1, (P, d))
    theta = np.array([0.3, 0.3, 0.3, 1.0, 0.1, 1.0])
    dc = None
    if world > 1:
        grid = os.environ.get("B200GP_C4_GRID")                 # e.g. "4x2"; default: dist.default_grid (2 x 4 on 8 GPUs)
        dc = dist.DistContext(ctx=ctx, rank=rank, world=world, grid=tuple(int(v) for v in grid.split("x")) if grid else None)
        nb = int(os.environ.get("B200GP_C4_NB", nb))

    def timed(fn):
        fn()                                   # warm-up: allocations, tile lists, NCCL channels
        ms, fac = [], []
        for _ in range(steps):
            barrier_sync(td, local)
            r = fn()
            t = ctx.last_timing()
            ms.append(t["total_ms"])
            fac.append(t["potrf_ms"])
        return r, max_over_ranks(td, local, float(np.mean(ms))), max_over_ranks(td, local, float(np.mean(fac)))

    if world > 1:
        r, ms, fac = timed(lambda: dc.posterior("RBF", X, y, Xn, theta, nb=nb))
        grid = f"{dc.grid[0]}x{dc.grid[1]}"
    else:
        def one_gpu():
            ctx.set_option("drop_factor_cache", 1)          # same X and theta every step: without this the factor is reused
            return ctx.posterior("RBF", X, y, Xn, theta[None], want=("mean", "var"))
        r, ms, fac = timed(one_gpu)
        r = {"mean": r["mean"][0], "var": r["var"][0], "info": int(r["info"][0])}
        grid = "1x1 (single-GPU entry point)"
    assert r["info"] == 0 and np.isfinite(r["mean"]).all() and (r["var"] > 0).all()
    flops = N ** 3 / 3 + N * N * (P + 1)
    out["c4_blockcyclic"] = {"workload": "exactgp_rbf_N32768_d3_P1024", "scaling": "strong", "n_gpus": world, "grid": grid, "tile": nb,
                             "ms_per_posterior": ms, "posteriors_per_s": 1e3 / ms, "factorisation_ms": fac if world > 1 else None,
                             "fp64_equiv_tflops_aggregate": flops / ms / 1e9, "checksum_mean": float(np.abs(r["mean"]).sum()),
                             "collectives": "column-comm broadcast of L_kk^-T, row-comm broadcast + column-comm all-gather of the panel "
                                            "(NCCL inside libb200gp.so), final all-reduce of mean / var" if world > 1 else "none"}
    # ---- c5
    N, d, M, P = 262144, 2, 4096, 4096
    rng = np.random.default_rng(6)
    X = rng.uniform(0, 1, (N, d))
    y = np.sin(9 * X[:, 0]) * np.cos(7 * X[:, 1]) + 0.05 * rng.standard_normal(N)
    Xu = X[rng.choice(N, M, replace=False)]
    Xn = rng.uniform(0, 1, (P, d))
    theta = np.array([0.2, 0.2, 1.0, 0.05, 1.0])
    if world > 1:
        lo, hi = rank * N // world, (rank + 1) * N // world
        r, ms, _ = timed(lambda: dc.sparse_posterior("Matern", Xu, X[lo:hi], y[lo:hi], Xn, theta, jitter=1e-5))
        allred = max_over_ranks(td, local, ctx.last_timing()["trsm_ms"])
    else:
        r, ms, _ = timed(lambda: ctx.sparse_posterior("Matern", Xu, X, y, Xn, theta, jitter=1e-5, want=("mean", "var")))
        allred = None
    assert r["info"] == 0 and np.isfinite(r["mean"]).all()
    flops = 2.0 * M * M * N + 2.0 * M ** 3 / 3 + 2.0 * M * M * (P + 1)
    out["c5_sharded_sparse"] = {"workload": "visparsegp_matern_N262144_d2_M4096_P4096", "scaling": "strong", "n_gpus": world,
                                "ms_per_posterior": ms, "posteriors_per_s": 1e3 / ms, "allreduce_ms": allred,
                                "fp64_equiv_tflops_aggregate": flops / ms / 1e9, "checksum_mean": float(np.abs(r["mean"]).sum()),
                                "collectives": "one all-reduce of the M x M statistics (134 MB) inside libb200gp.so" if world > 1 else "none"}
    if dc is not None:
        dc.close()
    return out


def run_reference_arm(args, rank, budget_s=270.0):
    """--impl reference: the reference's own CPU formulation (gpax cannot be imported: JAX absent; the oracle is
    its op-for-op NumPy restatement), all host threads, same config / metric / unit.

    MEASURED, not extrapolated: every timed step is one whole posterior at the workload's own N = 16384 (explicit
    inverse as gp.py:271, ~1-3 minutes on the box's host cores).  The driver's `--steps K` cannot be honoured at that
    cost (K = 20 would take an hour), so the arm times as many whole posteriors as fit `budget_s` (at least one,
    at most K) and reports that count in `steps`, the request in `steps_requested`; `ms_per_step` x `steps` is the real
    timed region.  Warm-up is one posterior at N = 2048 (thread pool and page faults; the N = 16384 arrays are touched
    before the timer starts)."""
    if rank != 0:
        return
    w = WORKLOAD
    import oracle
    cores = os.cpu_count()
    params = {"k_length": np.full(w["d"], w["ell"]), "k_scale": w["scale"], "noise": w["noise"]}
    X, y, Xn, _ = make_inputs(0)
    oracle.exact_posterior(X[:2048], y[:2048], Xn, params, "RBF", jitter=w["jitter"])           # warm-up
    times = []
    t_start = time.perf_counter()
    while len(times) < max(1, args.steps):
        t0 = time.perf_counter()
        mean, cov = oracle.exact_posterior(X, y, Xn, params, "RBF", jitter=w["jitter"])
        times.append(time.perf_counter() - t0)
        assert np.isfinite(mean).all() and cov.shape == (w["P"], w["P"])
        if (time.perf_counter() - t_start) + times[-1] > budget_s:
            break
    t = float(np.mean(times))
    val = 1.0 / t
    line = {"impl": "reference", "metric": "gp_posteriors_per_s_N16384", "value": val, "unit": "posteriors/s",
            "n_gpus": args.gpus, "steps": len(times), "steps_requested": args.steps, "warmup": 1,
            "warmup_requested": args.warmup, "ms_per_step": t * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": w["name"], "N": w["N"], "d": w["d"], "P": w["P"], "kernel": w["kernel"],
                       "measured_N": w["N"], "extrapolated": False},
            "steps_note": f"each step = one whole N={w['N']} posterior ({t:.1f} s); {len(times)} of the {args.steps} requested "
                          f"steps fit the {budget_s:.0f} s budget; warm-up = one N=2048 posterior",
            "cpu_baseline": {"value": val, "unit": "posteriors/s", "cores": cores, "kind": "port",
                             "sample": f"{len(times)} whole posterior(s) at N={w['N']} P={w['P']}, {t:.1f} s each, no scaling; "
                                       "oracle.exact_posterior = NumPy restatement of gpax ExactGP.get_mvn_posterior "
                                       "(explicit inverse, gp.py:271); gpax itself needs JAX, which is not installable here"},
            "e2e": {"value": val, "unit": "posteriors/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--draws", type=int, default=None, help="posterior draws per step (default 8)")
    ap.add_argument("--no-dist", action="store_true", help="skip the c4 / c5 exchange-step workloads")
    ap.add_argument("--opt", action="append", default=[], help="library option key=value (experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's mean and var to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    if args.impl == "reference":
        run_reference_arm(args, int(os.environ.get("RANK", "0")))
        return

    rank, world, local, td = dist_setup(args.gpus)
    from gpax_b200 import _ffi as ffi
    w = WORKLOAD
    ctx = ffi.Context(local)
    ctx.set_option("streams", args.streams)
    for kv in args.opt:
        k_, v_ = kv.split("=")
        ctx.set_option(k_, int(v_))
    if args.draws:
        WORKLOAD["S"] = args.draws
    X, y, Xn, theta = make_inputs(rank)
    N, d, P, S = w["N"], w["d"], w["P"], w["S"]
    flags_out = ffi.OUT_MEAN | ffi.OUT_VAR

    # ---- device-resident arm ("value")
    dX, dy, dXn, dth = ctx.to_device(X), ctx.to_device(y), ctx.to_device(Xn), ctx.to_device(theta)
    dmean, dvar = ctx.alloc((S, P)), ctx.alloc((S, P))
    info = np.zeros(S, dtype=np.int32)
    tim = ffi.Timing()

    def step_device():
        ctx._check(ctx.lib.b2gp_posterior(ctx.h, ffi.KIND[w["kernel"]], dX.ptr, N, dy.ptr, 0, dXn.ptr, P, d, S, dth.ptr, 0,
                                          w["jitter"], flags_out | ffi.FLAG_DEVICE_PTRS, dmean.ptr, dvar.ptr, None, None, 0,
                                          None, info.ctypes.data, None))
        t = ctx.last_timing()
        HOST_MS.append(t["host_enqueue_ms"])
        return t["total_ms"], t["launches"]

    for _ in range(max(args.warmup, 3)):
        step_device()
    assert (info == 0).all(), f"factorisation failed in warm-up: info={info}"
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    barrier_sync(td, local)
    ctx.sync()
    t0 = time.perf_counter()
    dev_ms, launches = 0.0, 0
    for _ in range(args.steps):
        ms, nl = step_device()
        dev_ms += ms
        launches += nl
    ctx.sync()
    barrier_sync(td, local)
    t1 = time.perf_counter()
    clocks = sampler.stop(t0, t1)
    if args.dump_outputs:
        assert (info == 0).all(), f"factorisation failed in the last timed step: info={info}"
        dump_outputs(args.dump_outputs, {"mean": dmean.download(), "var": dvar.download()},
                     f"_rank{rank}" if world > 1 else "")
    wall_ms = (t1 - t0) * 1e3
    dev_ms = max_over_ranks(td, local, dev_ms)
    wall_ms = max_over_ranks(td, local, wall_ms)
    value = world * S * args.steps / (dev_ms / 1e3)

    # ---- end-to-end arm: host (pinned) buffers through the C-ABI
    hX, hy, hXn, hth = ctx.pinned((N, d)), ctx.pinned((N,)), ctx.pinned((P, d)), ctx.pinned((S, d + 3))
    hX[:], hy[:], hXn[:], hth[:] = X, y, Xn, theta
    hmean, hvar = ctx.pinned((S, P)), ctx.pinned((S, P))

    def step_host():
        ctx._check(ctx.lib.b2gp_posterior(ctx.h, ffi.KIND[w["kernel"]], hX.ctypes.data, N, hy.ctypes.data, 0, hXn.ctypes.data,
                                          P, d, S, hth.ctypes.data, 0, w["jitter"], flags_out, hmean.ctypes.data,
                                          hvar.ctypes.data, None, None, 0, None, info.ctypes.data, None))
    step_host()
    barrier_sync(td, local)
    ctx.sync()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    ctx.sync()
    barrier_sync(td, local)
    e2e_s = max_over_ranks(td, local, time.perf_counter() - t0)
    e2e_value = world * S * args.steps / e2e_s
    assert np.isfinite(hmean).all() and (hvar > 0).all()
    h2d = X.nbytes + y.nbytes + Xn.nbytes + theta.nbytes
    d2h = hmean.nbytes + hvar.nbytes + info.nbytes

    # ---- one posterior alone (S = 1, host buffers): the latency a viGP.predict / get_mvn_posterior caller sees, with the
    # library's own phase clock (CUDA events inside the call).  Not part of `value`; rank 0 of the N=1 run only.
    single = None
    if rank == 0 and world == 1:
        lat = []
        for _ in range(4):
            ctx.set_option("drop_factor_cache", 1)
            t0 = time.perf_counter()
            o1 = ctx.posterior(w["kernel"], X, y, Xn, theta[:1], jitter=w["jitter"], want=("mean", "var"), timing=True)
            lat.append(((time.perf_counter() - t0) * 1e3, o1["timing"]))
        lat.sort(key=lambda r: r[0])
        ms1, t1_ = lat[len(lat) // 2 - 1]
        single = {"ms": ms1, "posteriors_per_s": 1e3 / ms1, "launches": int(t1_["launches"]),
                  "phases_ms": {k_: round(float(v_), 3) for k_, v_ in t1_.items() if k_.endswith("_ms")},
                  "note": "S=1, one stream: the fp64 chain of the diagonal blocks is exposed here and hidden in `value` by 8 draws in flight"}

    for a in (dX, dy, dXn, dth, dmean, dvar):
        a.free()

    def exchange_workloads(line):
        """c4 / c5 (every rank takes part).  They come AFTER the headline measurement and under a watchdog: a hang in a
        collective must not cost the bench line -- rank 0 then prints the line without these extras and the ranks exit."""
        if args.no_dist:
            return {}

        def bail():
            if rank == 0 and line is not None:
                line["dist_error"] = "c4 / c5 workloads did not finish within 600 s"
                emit(json.dumps(line))
            os._exit(0)
        wd = threading.Timer(600.0, bail)
        wd.daemon = True
        wd.start()
        try:
            return dist_workloads(ctx, ffi, rank, world, local, td)
        except Exception as e:  # noqa: BLE001
            return {"dist_error": repr(e)[:400]}
        finally:
            wd.cancel()

    if rank != 0:
        exchange_workloads(None)
        if td is not None:
            td.destroy_process_group()
        return
    # ---- roofline of the dominant kernel
    dom = measure_dominant_kernel(ctx, ffi)
    try:
        peak64 = measure_fp64_peak(local)
        peak_src = "cuBLAS DGEMM 8192^3 (torch.matmul fp64) measured in this run; MEASURED_PEAKS.json has no fp64 figure"
    except Exception as e:  # noqa: BLE001
        peak64, peak_src = 35.5, f"fallback 35.5 TFLOP/s (cuBLAS DGEMM measured on this pool, profiles/); live measure failed: {e!r}"
    peak = peak64
    # int8 tensor peak: MEASURED in this run by a bare tcgen05.mma kind::i8 loop (oz_i8_peak_kernel: M128 N256 K32, operands
    # resident in shared memory, every SM) -- MEASURED_PEAKS.json has no int8 figure, and 2 x its cuBLAS bf16 number
    # (3.46 POP/s, last round's denominator) understates the pipe, which the probe runs at 4.5 POP/s
    int8_peak, int8_src = None, None
    try:
        import ctypes as C_
        fn = ctx.lib.b2gp_debug_i8_peak
        fn.restype = C_.c_int
        fn.argtypes = [C_.c_void_p, C_.c_int, C_.c_int, C_.POINTER(C_.c_double), C_.POINTER(C_.c_double)]
        tops, pms = C_.c_double(), C_.c_double()
        if fn(ctx.h, 32768, 3, C_.byref(tops), C_.byref(pms)) == 0:
            int8_peak, int8_src = float(tops.value), "measured in this run: oz_i8_peak_kernel (bare tcgen05.mma kind::i8 M128 N256 K32 loop on all SMs)"
    except Exception:  # noqa: BLE001
        pass
    mp_bf16 = None
    try:
        mp_bf16 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
    except Exception:  # noqa: BLE001
        pass
    if int8_peak is None:
        int8_peak, int8_src = 2.0 * (mp_bf16 or 1590.0), "2 x bf16 tensor peak (MEASURED_PEAKS.json or the B200_PROFILING.md fallback): the int8 probe failed"
    traffic = None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "dominant_kernel.json")))
        traffic = prof.get("dram_bytes_per_launch")
    except Exception:  # noqa: BLE001
        pass
    oz = dom["tcgen05_i8"]
    int8_tops = dom["int8_ops_per_launch"] / oz["ms"] / 1e9
    flops_step = S * (N ** 3 / 3 + N * N * (P + 1) + 4 * N * P)
    line = {
        "metric": "gp_posteriors_per_s_N16384", "value": value, "unit": "posteriors/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": w["name"], "N": N, "d": d, "P": P, "kernel": w["kernel"], "draws_per_step": S,
                   "outputs": "mean+diag var", "streams": args.streams, "parallelism": f"draw-parallel x{world}",
                   "l2": "inputs larger than L2: each draw rebuilds and factors a 2 GiB K (L2 = 126 MB)"},
        "wall_ms_per_step": wall_ms / args.steps,
        "host_enqueue_ms_per_step": float(np.mean(HOST_MS[-args.steps:])),
        "fp64_tflops_step": world * flops_step * args.steps / (dev_ms / 1e3) / 1e12,
        "frac_of_chol_roofline_N3_3": (world * S * args.steps * N ** 3 / 3 / (dev_ms / 1e3) / 1e12) / (world * peak),
        "frac_of_chol_roofline_2N3_3": (world * S * args.steps * 2 * N ** 3 / 3 / (dev_ms / 1e3) / 1e12) / (world * peak),
        "e2e": {"value": e2e_value, "unit": "posteriors/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "clocks": clocks,
        # dominant kernel: oz_mma_kernel<S> (int8 tcgen05.mma into TMEM, TMA-fed).  Algorithmic work of the launch =
        # S(S+1)/2 digit-plane-pair int8 GEMMs of the 8192x8192 lower half at k = 8192; denominator = int8 dense tensor peak.
        "roofline": {"bound": "tensor", "achieved": int8_tops, "peak": int8_peak, "unit": "TOP/s (int8)", "frac": int8_tops / int8_peak,
                     "traffic": traffic, "kernel": f"oz_slice_kernel<{dom['planes']}> + oz_mma_kernel<{dom['planes']},2> (UTCIMMA M128 N<=256 K32 over stacked digit planes, TMEM "
                     "accumulators, CTA-pair TMA multicast, 32B-swizzle stages; SYRK 8192x8192 k=8192 lower)", "int8_ops_per_launch": dom["int8_ops_per_launch"],
                     "ms_per_launch": oz["ms"], "peak_source": int8_src,
                     "frac_of_2x_measured_bf16": (int8_tops / (2.0 * mp_bf16)) if mp_bf16 else None,
                     "fp64_equiv_tflops": oz["fp64_equiv_tflops"], "fp64_equiv_over_cublas_dgemm": oz["fp64_equiv_tflops"] / peak64,
                     "digit_planes": dom["planes"], "plane_pairs": dom["pairs"]},
        # the fp64 DMMA kernel (gemm_tma_kernel) that the int8 path replaces for large updates, same launch
        "roofline_dmma": {"bound": "tensor", "achieved": dom["dmma"]["fp64_equiv_tflops"], "peak": peak64, "unit": "TFLOP/s",
                          "frac": dom["dmma"]["fp64_equiv_tflops"] / peak64, "ms_per_launch": dom["dmma"]["ms"],
                          "kernel": "gemm_tma_kernel<3,2> (DMMA.8x8x4, TMA + mbarrier) + 64x64 tail launch", "peak_source": peak_src},
    }
    if single is not None:
        line["single_posterior"] = single
    line.update(exchange_workloads(line))
    if not args.no_cpu_baseline and world == 1:      # a reported baseline of the N=1 line only
        line["cpu_baseline"] = cpu_baseline()
    emit(json.dumps(line))
    if td is not None:
        td.destroy_process_group()


if __name__ == "__main__":
    main()
