#!/usr/bin/env python
"""bench.py -- throughput of the B200 SVGP-ELBO / Laplace hot path, FP64.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c4|c2|c5|c5mb|c3|c1|...]

Default workload = BASELINE.json configs[3] ("C4": SVGP PoissonLikelihood, SqExponential, N = 1e7, D = 8, M = 1024, Float64), the
configuration the headline metric is quoted on.  A "step" is one full `elbo` + all-gradients evaluation (agp_svgp_elbo_grad
through the C ABI) over the whole synthetic data set.  With N > 1 ranks (torchrun, one process per GPU) the points are sharded
contiguously over the ranks and the partial sums are combined by one ncclAllReduce per step inside the library.  The other
BASELINE.json configurations are reachable with --workload: c2 (Bernoulli GH-20, Matern52, N = 1e6, M = 512), c5 (Gaussian,
N = 1e8, D = 16, M = 2048, full sweep, data generated on the device), c5mb (one 2^20-point minibatch per rank of the same
model, num_data = 1e8), c3 (LaplaceApproximation, N = 8192; a step is one `approx_lml`, i.e. one Newton loop) and c1 (the
a-regression example: minibatches of 100 points, M = 20 / 50).

One JSON line is printed by rank 0 (DESIGN.md "Measurement" explains every key):
  value     metric with the inputs already resident in HBM when the timed region starts (profiling events off)
  e2e       the same metric through the same C-ABI calls with HOST (pinned) x, y: every step uploads the shard
            (agp_dataset_upload), evaluates, and reads ELBO + gradients back
  roofline  dominant kernel class: algorithmic FP64 flop / CUDA-event launch time (a separate, profiled pass of the same steps)
            against the FP64 DMMA issue peak MEASURED IN THIS RUN (agp_fp64_peak; MEASURED_PEAKS.json has no FP64 entry)
  correctness  N > 1: the first 2^18 points evaluated sharded (NCCL path) and by rank 0 alone, ELBO and every gradient buffer
            compared; N = 1: the same buffers against the CPU restatement on the cpu_baseline sample
  cpu_baseline  the NumPy/OpenBLAS restatement of the reference's op sequence (oracle/), timed on this box's host cores on a
            bounded sample (rank 0, N = 1 only)

`--impl reference` times that CPU restatement alone (Julia is not installed, so the reference itself cannot run; see
DESIGN.md) and prints the same line with "impl": "reference".
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "SVGP ELBO+grad points/sec (FP64)"
UNIT = "points/s"

# Fallback denominators, used only if the in-run measurement fails: FP64 DMMA issue peak and cuBLAS DGEMM 8192^3 measured on this
# pool's B200 in round 1 (tools/fp64_peak.cu, tools/dgemm_peak.py -> profiles/r01_*).
FP64_PEAK_TFLOPS_DMMA = 37.1
FP64_PEAK_TFLOPS_DGEMM = 35.5

# dram__bytes_read.sum + dram__bytes_write.sum per launch of the sweep kernels at the C4 chunk shape (M = 1024, D = 8, 151 552 points per
# launch), from the `ncu --set full` captures summarised in profiles/ (r01x: round 1; refreshed by the round-2 captures)
NCU_TRAFFIC_BYTES_C4 = {"trsm_kuf_fwd": 1.753e9 + 1.336e9, "gemm_BC": 4.599e9 + 2.476e9}

WORKLOADS = {
    # BASELINE.json configs[3] (the configuration `metric` is quoted on)
    "c4": dict(label="C4 SVGP Poisson(exp) analytic, SqExponential, N=1e7, D=8, M=1024, FP64", N=10_000_000, D=8, M=1024, kind="se",
               lik="poisson_exp", method="default", seed=4, lengthscale=math.sqrt(8.0), variance=1.0, jitter=1e-6),
    # SURVEY.md section 8(d) variants of C4: Gauss-Hermite(20) instead of the analytic Poisson expectation; Matern52 kernel
    "c4gh": dict(label="C4 variant: SVGP Poisson(exp) Gauss-Hermite(20), SqExponential, N=1e7, D=8, M=1024, FP64", N=10_000_000, D=8, M=1024,
                 kind="se", lik="poisson_exp", method="gauss_hermite", seed=4, lengthscale=math.sqrt(8.0), variance=1.0, jitter=1e-6),
    "c4m52": dict(label="C4 variant: SVGP Poisson(exp) analytic, Matern52, N=1e7, D=8, M=1024, FP64", N=10_000_000, D=8, M=1024,
                  kind="matern52", lik="poisson_exp", method="default", seed=4, lengthscale=math.sqrt(8.0), variance=1.0, jitter=1e-6),
    # BASELINE.json configs[1]
    "c2": dict(label="C2 SVGP Bernoulli GH-20, Matern52, N=1e6, D=8, M=512, FP64", N=1_000_000, D=8, M=512, kind="matern52",
               lik="bernoulli_logit", method="default", seed=2, lengthscale=math.sqrt(8.0), variance=1.0, jitter=1e-6),
    # BASELINE.json configs[4]: the full sweep over N = 1e8 points (strong scaling over the ranks), generated on the device
    "c5": dict(label="C5 SVGP Gaussian, SqExponential, N=1e8 full sweep, D=16, M=2048, FP64", N=100_000_000, D=16, M=2048, kind="se",
               lik="gaussian", method="default", seed=5, lengthscale=4.0, variance=1.0, jitter=1e-6, device_gen=True, long_step=True),
    # ... and one rank-step of its minibatch mode (2^20 points per rank, num_data = 1e8): weak scaling
    "c5mb": dict(label="C5 minibatch SVGP Gaussian, SqExponential, B=2^20/rank, num_data=1e8, D=16, M=2048, FP64", N=1 << 20, D=16,
                 M=2048, kind="se", lik="gaussian", method="default", seed=5, lengthscale=4.0, variance=1.0, jitter=1e-6,
                 num_data=1e8, weak=True),
    # BASELINE.json configs[0]: examples/a-regression/script.jl -- 300 epochs of 100 minibatches (100 points each) with M = 20 inducing points
    # (the script's value; BASELINE.json says 50: reported as well).  Latency-bound: a step here is ONE EPOCH = 100 minibatch evaluations.
    "c1": dict(label="C1 a-regression SVGP Gaussian, SqExponential, N=1e4, D=1, minibatch 100, num_data=N, FP64 (one epoch = 100 ELBO+grad evaluations per step)",
               N=10_000, D=1, M=20, small=True),
    # BASELINE.json configs[2]: LaplaceApproximation, Bernoulli-logit, dense N = 8192 latent GP (replicas only: see DESIGN.md)
    "c3": dict(label="C3 Laplace Bernoulli-logit, SqExponential, N=8192, D=2, FP64 (one approx_lml = one Newton loop per step)", N=8192, D=2,
               laplace=True),
}

BLOCK = 1 << 20  # rows per generation block: the global data set is independent of the rank count


def flops_per_point(M: int, D: int) -> float:
    """SURVEY.md section 8(d): algorithmic flop per point for ELBO + gradient (the reference's operation count)."""
    return 6.0 * M * M + 6.0 * M * D


# algorithmic flop per point of each kernel class (DESIGN.md "Kernels").  The reference's reverse pass has two M x N . N x M products
# (dB and dLk, M^2 each); here one symmetric rank-N update G += As A^T serves both, and it is counted with the standard SYRK
# figure M^2 so that its roofline fraction is not inflated: the classes therefore add up to flops_per_point minus that saved M^2.
def class_flops_per_point(M: int, D: int) -> dict:
    return {"trsm_kuf_fwd": M * M + 2.0 * M * D, "gemm_BtA": 1.0 * M * M, "gemm_BC": 1.0 * M * M, "trsm_bwd": 1.0 * M * M,
            "syrk_G": 1.0 * M * M, "kgrad": 4.0 * M * D}


SAVED_BY_ALGEBRA = lambda M, D: 1.0 * M * M  # noqa: E731


def executed_flops_per_point(M: int, D: int) -> float:
    """What the device code executes per point: the sum of the kernel classes (5 M^2 + 6 M D)."""
    return flops_per_point(M, D) - SAVED_BY_ALGEBRA(M, D)


def gen_rows(w: dict, lo: int, hi: int, wvec: np.ndarray):
    """Rows [lo, hi) of the synthetic data set (SURVEY.md section 8(d) recipe), block-seeded."""
    D = w["D"]
    X = np.empty((hi - lo, D))
    y = np.empty(hi - lo)
    b0, b1 = lo // BLOCK, (hi - 1) // BLOCK
    for b in range(b0, b1 + 1):
        rng = np.random.default_rng([w["seed"], b])
        Xb = rng.standard_normal((BLOCK, D))
        g = np.sin(Xb @ wvec)
        if w["lik"] == "poisson_exp":
            yb = rng.poisson(np.exp(0.5 * g)).astype(np.float64)
        elif w["lik"] == "bernoulli_logit":
            yb = (rng.random(BLOCK) < 1.0 / (1.0 + np.exp(-2.0 * g))).astype(np.float64)
        else:
            yb = g + 0.1 * rng.standard_normal(BLOCK)
        s, e = max(lo, b * BLOCK), min(hi, (b + 1) * BLOCK)
        X[s - lo:e - lo] = Xb[s - b * BLOCK:e - b * BLOCK]
        y[s - lo:e - lo] = yb[s - b * BLOCK:e - b * BLOCK]
    return X, y


def gen_rows_device(w: dict, lo: int, hi: int, wvec: np.ndarray, device):
    """The same recipe generated on the device (C5: 1e8 x 16 doubles are 12.8 GB -- SURVEY.md section 8(d) asks for per-shard device
    generation); block-seeded torch Philox streams, so the global data set is again independent of the rank count."""
    import torch

    D = w["D"]
    X = torch.empty((hi - lo, D), dtype=torch.float64, device=device)
    y = torch.empty((hi - lo,), dtype=torch.float64, device=device)
    wv = torch.from_numpy(wvec).to(device)
    g = torch.Generator(device=device)
    for b in range(lo // BLOCK, (hi - 1) // BLOCK + 1):
        g.manual_seed(1_000_003 * w["seed"] + b)
        Xb = torch.randn((BLOCK, D), dtype=torch.float64, device=device, generator=g)
        nb = torch.randn((BLOCK,), dtype=torch.float64, device=device, generator=g)
        yb = torch.sin(Xb @ wv) + 0.1 * nb
        s, e = max(lo, b * BLOCK), min(hi, (b + 1) * BLOCK)
        X[s - lo:e - lo] = Xb[s - b * BLOCK:e - b * BLOCK]
        y[s - lo:e - lo] = yb[s - b * BLOCK:e - b * BLOCK]
    return X, y


def make_params(w: dict):
    """Replicated (tiny) inputs: Z, m, Lq, kernel."""
    rng = np.random.default_rng([w["seed"], 10_000_019])
    D, M = w["D"], w["M"]
    wvec = rng.standard_normal(D)
    X0, _ = gen_rows(w, 0, M, wvec)
    Z = X0 + 1e-3 * rng.standard_normal((M, D))
    m = 0.1 * rng.standard_normal(M)
    A = 0.5 * np.eye(M) + 0.01 * np.tril(rng.standard_normal((M, M)))
    A[np.diag_indices(M)] = np.abs(np.diag(A))
    return wvec, Z, m, A


def oracle_objects(w, Z, m, A):
    from oracle import kernels as ok, likelihoods as ol, svgp as osv

    k = ok.Kernel(w["kind"], w["variance"], np.array([1.0 / w["lengthscale"]]), 0.0)
    s = osv.SVGP(k, Z, m, A, jitter=w["jitter"])
    return s, ol.Likelihood(w["lik"], 0.01), ol.Expectation(w["method"], 20)


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # pragma: no cover
        return os.cpu_count() or 1


def time_oracle(w, Z, m, A, X, y, reps: int, num_data: float, chunk: int = 65536):
    """points/s of the CPU restatement on the given rows (OpenBLAS threads = host cores); also returns its last result."""
    from threadpoolctl import threadpool_limits

    from oracle import svgp as osv

    s, lik, ex = oracle_objects(w, Z, m, A)
    times, res = [], None
    with threadpool_limits(limits=host_threads()):
        for _ in range(reps):
            t0 = time.perf_counter()
            res = osv.elbo_and_grad(s, X, y, lik, ex, num_data=num_data, chunk=chunk)
            times.append(time.perf_counter() - t0)
    return len(y) / statistics.median(times), times, res


def svgp_config(w, N_total, world, n_local):
    return {"workload": w["label"], "N": N_total, "M": w["M"], "D": w["D"], "points_per_rank": n_local,
            "parallelism": f"dp{world} (N-sharded, 1 ncclAllReduce/step)",
            "l2": "no flush needed: every step streams the X shard plus >1 GB of per-chunk scratch, far beyond the 126 MB L2"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(gpu_index)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        for line in self.f.read().splitlines():
            c = [t.strip() for t in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            load = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] or sm
            out = {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm), "reasons": sorted(reasons)}
        return out


# ---------------------------------------------------------------------------------------------------------------------
# --impl reference: the CPU restatement of the reference's op sequence on the host cores
# ---------------------------------------------------------------------------------------------------------------------
def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if w.get("laplace"):
        return run_reference_laplace(args, w)
    if w.get("small"):
        return run_reference_c1(args, w)
    wvec, Z, m, A = make_params(w)
    cores = host_threads()
    Xp, yp = gen_rows(w, 0, 8192, wvec)
    pps, _, _ = time_oracle(w, Z, m, A, Xp, yp, 1, w["N"], chunk=8192)  # pilot
    budget = 150.0 / max(1, args.steps + args.warmup)
    n_sample = int(min(262144, max(8192, 2 ** int(math.log2(max(1.0, pps * min(budget, 20.0)))))))
    from threadpoolctl import threadpool_limits

    from oracle import svgp as osv

    s, lik, ex = oracle_objects(w, Z, m, A)
    X, y = gen_rows(w, 0, n_sample, wvec)
    num_data = float(w.get("num_data", w["N"]))
    with threadpool_limits(limits=cores):
        for _ in range(args.warmup):
            osv.elbo_and_grad(s, X, y, lik, ex, num_data=num_data, chunk=65536)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            osv.elbo_and_grad(s, X, y, lik, ex, num_data=num_data, chunk=65536)
        dt = time.perf_counter() - t0
    value = n_sample * args.steps / dt
    sample = f"rows [0,{n_sample}) of the workload per step, chunked 65536, NumPy/SciPy OpenBLAS threads={cores}"
    world = args.gpus
    N_total = w["N"] * world if w.get("weak") else w["N"]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak" if w.get("weak") else "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": svgp_config(w, N_total, world, (N_total + world - 1) // world),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "gflops": value * flops_per_point(w["M"], w["D"]) / 1e9},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference-algorithm CPU restatement (oracle/, NumPy + OpenBLAS); Julia is not installed so ApproximateGPs.jl itself cannot run"}
    print(json.dumps(line), flush=True)


LAPLACE_METRIC = "Laplace approx_lml Newton iterations/sec (N=8192, FP64)"
LAPLACE_UNIT = "iterations/s"


def laplace_flops_per_iteration(n: int) -> float:
    """SURVEY.md section 8(d): one Newton iteration = one Cholesky of B (n^3/3) + 6 n^2 (B assembly, two symv, two triangular solves)."""
    return n**3 / 3.0 + 6.0 * n * n


def c3_problem(n: int):
    rng = np.random.default_rng(3)
    X = rng.uniform(0, 10, size=(n, 2))
    y = (rng.random(n) < 1 / (1 + np.exp(-3 * np.sin(X[:, 0])))).astype(np.float64)
    return X, y


def time_oracle_laplace(n_cpu: int, reps: int):
    from threadpoolctl import threadpool_limits

    from oracle import kernels as ok, laplace as olap, likelihoods as ol

    X, y = c3_problem(8192)
    K = ok.kernelmatrix(ok.Kernel("se", 1.0, np.array([1.0])), X[:n_cpu]) + 1e-8 * np.eye(n_cpu)
    ts, steps = [], 0
    with threadpool_limits(limits=host_threads()):
        for _ in range(reps):
            t0 = time.perf_counter()
            _, _, steps = olap.laplace_f_and_lml(ol.Likelihood("bernoulli_logit"), y[:n_cpu], K)
            ts.append(time.perf_counter() - t0)
    return statistics.median(ts), steps


def run_reference_laplace(args, w):
    n, n_cpu, cores = w["N"], 2048, host_threads()
    for _ in range(min(args.warmup, 1)):
        time_oracle_laplace(n_cpu, 1)
    t, steps = time_oracle_laplace(n_cpu, max(1, args.steps))
    iters = steps + 1  # the loop's iterations plus the recomputation at f_opt (Laplace.jl:144)
    gflops = laplace_flops_per_iteration(n_cpu) * iters / t / 1e9
    value = gflops * 1e9 / laplace_flops_per_iteration(n)  # iterations/s at N = 8192 at the flop rate measured at n_cpu
    sample = (f"the same recipe at n={n_cpu} ({iters} Newton iterations, {t:.2f} s, {gflops:.1f} GFLOP/s), extrapolated to N={n} by the flop count "
              f"n^3/3 + 6 n^2; NumPy/SciPy OpenBLAS threads={cores}")
    line = {"impl": "reference", "metric": LAPLACE_METRIC, "value": value, "unit": LAPLACE_UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * iters / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": w["label"], "N": n, "D": w["D"], "parallelism": f"replicas x{args.gpus} (the path does not shard)"},
            "cpu_baseline": {"value": value, "unit": LAPLACE_UNIT, "cores": cores, "kind": "port", "sample": sample, "gflops": gflops},
            "e2e": {"value": value, "unit": LAPLACE_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference-algorithm CPU restatement (oracle/, NumPy + OpenBLAS); Julia is not installed so ApproximateGPs.jl itself cannot run"}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------------------------------
_JSON_OUT = None


def emit(line: dict):
    """The ONE JSON line of the contract, on the process's original stdout."""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_LIMIT_BYTES = 64 << 20


def snapshot(**arrays) -> dict:
    """float64 C-ordered copies of what a step returned: the passes after the timed one overwrite the same host buffers."""
    return {k: np.array(v, dtype=np.float64, order="C", ndmin=1) for k, v in arrays.items()}


def dump_outputs(path: str, arrays: dict):
    """--dump-outputs: the last timed step's results as DIR/<name>.npy, so that two builds run on the same seeded inputs can be
    compared output for output."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def setup_dist(args):
    # stdout carries exactly one JSON line.  NCCL logs to the process's stdout (its version banner at any NCCL_DEBUG level), so file
    # descriptor 1 is pointed at stderr for the lifetime of the process and the JSON line goes to a duplicate of the original stdout.
    # With more than one rank NCCL_DEBUG defaults to INFO: the communicator setup (rank count, rings, NVLS) lands on stderr.
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
        os.environ["NCCL_DEBUG"] = "INFO"  # (an inherited VERSION / WARN level would hide the communicator setup)
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return torch, dist, rank, world, local


def make_timer(torch, dist, world, stream):
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """K calls of fn bracketed by barrier + synchronize; device time (ms) on the library stream, max over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    return barrier, timed


def measure_fp64_peak(ctx):
    try:
        pk = ctx.fp64_peak()
        return pk["dmma"], pk["dfma"], "measured in this run (agp_fp64_peak: register-resident DMMA.8x8x4 / DFMA chains, best of 3)"
    except Exception as e:  # pragma: no cover
        return FP64_PEAK_TFLOPS_DMMA, None, f"round-1 measurement (in-run measurement failed: {e})"


def grad_struct(L, M, D):
    g_m, g_Lq, g_Z = np.zeros(M), np.zeros((M, M), order="F"), np.zeros((M, D))
    sc = np.zeros(4)
    g_ils = np.zeros(1)
    G = L.AgpSvgpGrads(L.dptr(g_m), L.dptr(g_Lq), L.dptr(g_Z), sc[0:1].ctypes.data_as(L.c_double_p), L.dptr(g_ils),
                       sc[1:2].ctypes.data_as(L.c_double_p), sc[2:3].ctypes.data_as(L.c_double_p), sc[3:4].ctypes.data_as(L.c_double_p))
    bufs = {"m": g_m, "Lq": g_Lq, "Z": g_Z, "variance": sc[0:1], "inv_lengthscale": g_ils, "lik_sigma2": sc[3:4]}
    return G, bufs


def rel_to_max(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def run_svgp(args, w):
    torch, dist, rank, world, local = setup_dist(args)
    import agp_b200 as agp
    from agp_b200 import _lib as L
    from agp_b200 import shard_range

    dev = torch.device("cuda", local)
    weak = bool(w.get("weak"))
    N_total = w["N"] * world if weak else w["N"]
    lo, hi = shard_range(N_total, rank, world)
    n_local = hi - lo
    D, M = w["D"], w["M"]
    wvec, Z, m, A = make_params(w)
    on_device = bool(w.get("device_gen"))
    host_bytes = 8 * n_local * (D + 1)
    keep_host = (not on_device) or host_bytes <= (8 << 30)  # the e2e leg needs a pinned host copy of the shard

    ctx = agp.Context(local)
    if world > 1:
        agp.attach_communicator(ctx, dist)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=dev)
    barrier, timed = make_timer(torch, dist, world, stream)
    peak_dmma, peak_dfma, peak_src = measure_fp64_peak(ctx)

    ds = agp.DeviceData(capacity=n_local, D=D, ctx=ctx)
    lib = ctx.lib
    Xh = yh = None
    if on_device:
        Xd, yd = gen_rows_device(w, lo, hi, wvec, dev)
        torch.cuda.synchronize()
        ds.upload_device(Xd.data_ptr(), n_local, yd.data_ptr())
        if keep_host:
            Xh = torch.empty((n_local, D), dtype=torch.float64).pin_memory()
            yh = torch.empty((n_local,), dtype=torch.float64).pin_memory()
            Xh.copy_(Xd)
            yh.copy_(yd)
        del Xd, yd
        torch.cuda.empty_cache()
    else:
        # host (pinned) copy of this rank's shard -- the e2e leg uploads it every step
        Xh = torch.empty((n_local, D), dtype=torch.float64).pin_memory()
        yh = torch.empty((n_local,), dtype=torch.float64).pin_memory()
        for s in range(0, n_local, BLOCK):
            e = min(n_local, s + BLOCK)
            Xb, yb = gen_rows(w, lo + s, lo + e, wvec)
            Xh[s:e] = torch.from_numpy(Xb)
            yh[s:e] = torch.from_numpy(yb)

    def upload():
        L.check(lib.agp_dataset_upload(ds.h, C.c_void_p(Xh.data_ptr()), n_local, D, L.POINT_MAJOR, C.c_void_p(yh.data_ptr()), L.Y_F64, L.HOST))
        ds.N = n_local

    base = {"se": agp.SqExponentialKernel, "matern32": agp.Matern32Kernel, "matern52": agp.Matern52Kernel}[w["kind"]]()
    f = agp.GP(w["variance"] * agp.with_lengthscale(base, w["lengthscale"]))
    sva = agp.SparseVariationalApproximation(f(Z, w["jitter"]), agp.MvNormal(m, chol_lower=A))
    lik = {"gaussian": agp.GaussianLikelihood(0.01), "bernoulli_logit": agp.BernoulliLikelihood(), "poisson_exp": agp.PoissonLikelihood()}[w["lik"]]
    pk = agp.PackedParams(sva, lik, agp.GaussHermiteExpectation(20) if w["method"] == "gauss_hermite" else None, args.dtype)
    f32 = args.dtype in ("f32", "f32_tc_solve")
    emu = args.dtype == "f64emu"
    G, gb = grad_struct(L, M, D)
    out = C.c_double()
    num_data = float(w.get("num_data", N_total))

    def step():
        L.check(lib.agp_svgp_elbo_grad(ctx.h, ds.h, 0, n_local, C.byref(pk.p), num_data, N_total, C.byref(out), C.byref(G)))
        return out.value

    # ---- device-resident leg (profiling events off: exactly the code path of the e2e leg) ---------------
    if not on_device:
        upload()
    # W >= 3 for every workload whose step is short; one C5 step is 1e8 points = 660 launch groups per kernel class (76 s on one GPU): the
    # given --warmup is honoured there (>= 1) and the line says so
    n_warm = max(1, args.warmup) if w.get("long_step") else max(3, args.warmup)
    for _ in range(n_warm):
        val = step()
    l0 = ctx.launch_count()
    clocks = ClockSampler(local) if rank == 0 else None
    ms = timed(step, args.steps)
    clk = clocks.stop() if clocks else {}
    launches = ctx.launch_count() - l0
    value = N_total * args.steps / (ms * 1e-3)
    last = snapshot(elbo=out.value, **{"grad_" + k: v for k, v in gb.items()})

    # ---- profiled pass: per-kernel-class CUDA-event times of the same steps (not part of `value`) -------
    psteps = 1 if w.get("long_step") else max(1, min(args.steps, 3))
    ctx.profile_read()
    ctx.profile(True)
    ms_prof = timed(step, psteps)
    prof = ctx.profile_read()
    ctx.profile(False)

    # ---- end-to-end leg: host buffers, upload + evaluate + read back every step ------------------------
    e2e = None
    if not args.no_e2e and Xh is not None:
        def e2e_step():
            upload()
            step()

        e2e_step()
        ms_e = timed(e2e_step, args.steps)
        p_bytes = 8 * (M * D + M + M * M + 4)
        g_bytes = 8 * (M + M * M + M * D + 6)
        e2e = {"value": N_total * args.steps / (ms_e * 1e-3), "unit": UNIT, "ms_per_step": ms_e / args.steps,
               "h2d_bytes_per_step": 8 * N_total * (D + 1) + world * p_bytes, "d2h_bytes_per_step": world * g_bytes}
    elif not args.no_e2e:
        e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
               "note": f"not run: the pinned host copy of one rank's shard would be {host_bytes / 2**30:.1f} GiB (run with more ranks)"}

    # ---- correctness at N > 1: the first n_check points, sharded over the ranks (NCCL path) vs rank 0 alone ----------
    correctness = None
    if world > 1 and not args.no_check:
        n_check = min(N_total, 1 << 18)
        clo, chi = shard_range(n_check, rank, world)
        if on_device:
            Xc_d, yc_d = gen_rows_device(w, 0, n_check, wvec, dev)
            Xc, yc = Xc_d.cpu().numpy(), yc_d.cpu().numpy()
            del Xc_d, yc_d
        else:
            Xc, yc = gen_rows(w, 0, n_check, wvec)
        dsc = agp.DeviceData(Xc[clo:chi], yc[clo:chi], ctx=ctx)
        Gs, gs = grad_struct(L, M, D)
        outs = C.c_double()
        L.check(lib.agp_svgp_elbo_grad(ctx.h, dsc.h, 0, chi - clo, C.byref(pk.p), num_data, n_check, C.byref(outs), C.byref(Gs)))
        dsc.close()
        if rank == 0:
            ctx1 = agp.Context(local)  # no communicator: a plain 1-rank evaluation of the same points
            ds1 = agp.DeviceData(Xc, yc, ctx=ctx1)
            G1, g1 = grad_struct(L, M, D)
            out1 = C.c_double()
            L.check(ctx1.lib.agp_svgp_elbo_grad(ctx1.h, ds1.h, 0, n_check, C.byref(pk.p), num_data, n_check, C.byref(out1), C.byref(G1)))
            errs = {k: rel_to_max(gs[k], g1[k]) for k in gs}
            correctness = {"what": f"rows [0,{n_check}) evaluated sharded over {world} ranks (one ncclAllReduce) vs by rank 0 alone, same C-ABI call",
                           "elbo_sharded": outs.value, "elbo_1rank": out1.value, "elbo_rel": abs(outs.value - out1.value) / abs(out1.value),
                           "grad_rel_to_max": errs, "grad_checksums_sharded": {k: float(np.sum(v)) for k, v in gs.items()},
                           "grad_checksums_1rank": {k: float(np.sum(v)) for k, v in g1.items()}, "tol": 1e-5 if f32 else 1e-11,
                           "note": "the two evaluations add the same per-point terms in a different order (per-rank partial sums, then the all-reduce); "
                                   "measured 0 on the ELBO and <= 2e-12 on the gradients"}
            correctness["ok"] = bool(correctness["elbo_rel"] < correctness["tol"] and max(errs.values()) < correctness["tol"])
            ds1.close()
            ctx1.close()
        barrier()

    if world > 1:
        lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(lt)
        launches = int(lt.item())

    if rank == 0:
        cf = class_flops_per_point(M, D)
        sweep = {k: v for k, v in prof.items() if v[1] > 0}
        tot_ms = sum(v[0] for v in sweep.values())
        kernels = {}
        for k, (kms, cnt) in sweep.items():
            ent = {"ms_per_step": kms / psteps, "share": kms / tot_ms if tot_ms else None, "launch_groups_per_step": cnt / psteps}
            if k in cf:
                ent["alg_tflops"] = cf[k] * n_local * psteps / (kms * 1e-3) / 1e12
                ent["frac_of_peak"] = ent["alg_tflops"] / peak_dmma
            kernels[k] = ent
        dom = max((k for k in sweep if k in cf), key=lambda k: sweep[k][0])
        dms, dcnt = sweep[dom]
        achieved = cf[dom] * n_local * psteps / (dms * 1e-3) / 1e12
        step_s = ms / args.steps * 1e-3
        alg_tf = flops_per_point(M, D) * N_total / step_s / 1e12 / world
        exe_tf = executed_flops_per_point(M, D) * N_total / step_s / 1e12 / world
        roof = {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peak_dmma, "unit": "TFLOP/s", "frac": achieved / peak_dmma,
                "traffic": NCU_TRAFFIC_BYTES_C4.get(dom) if (args.workload == "c4" and not args.n) else None,
                "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/)",
                "alg_bytes_per_launch": (8.0 * (D + 1) + 8.0 * M) * (n_local * psteps / dcnt) if dom == "trsm_kuf_fwd" else None,
                "avg_launch_ms": dms / dcnt, "alg_flop_per_launch": cf[dom] * n_local * psteps / dcnt,
                "peak_source": f"FP64 DMMA issue peak {peak_src}; DFMA {peak_dfma and round(peak_dfma, 2)} TFLOP/s; round-1 references: DMMA {FP64_PEAK_TFLOPS_DMMA}, "
                               f"cuBLAS DGEMM 8192^3 {FP64_PEAK_TFLOPS_DGEMM}; MEASURED_PEAKS.json has no FP64 entry",
                "kuf_trsm_stage": {"alg_tflops": kernels.get("trsm_kuf_fwd", {}).get("alg_tflops"), "frac_of_peak": kernels.get("trsm_kuf_fwd", {}).get("frac_of_peak")},
                "profiled_pass": {"steps": psteps, "ms_per_step": ms_prof / psteps},
                **({"note": "Float32 mode: the two triangular solves run on the INT8 tensor path and S2 / S4 / S6 on TF32; `achieved` and the fractions are "
                            "FP64-equivalent throughput set against the FP64 DMMA peak for comparison with the Float64 line, not a utilisation"} if f32 else {}),
                "whole_step": {"executed_tflops_per_gpu": exe_tf, "frac_of_fp64_peak_executed": exe_tf / peak_dmma,
                               "reference_equivalent_tflops_per_gpu": alg_tf,
                               "note": "executed = 5 M^2 + 6 M D flop per point (one SYRK serves the reference's two M x N . N x M products); "
                                       "reference-equivalent = SURVEY.md 8(d)'s 6 M^2 + 6 M D, a throughput figure, not a hardware utilisation"}}
        # the HBM-facing per-point stage (S3): algorithmic bytes 8 (5 + nb) per point against the measured copy bandwidth
        hbm_peak = None
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                hbm_peak = float(json.load(fh)["hbm_gbs"])
        except Exception:
            hbm_peak = 6650.0  # fallback of the profiling recipe
        pp_ms = sweep.get("perpoint", (0.0, 0))[0] / psteps
        nb_blocks = (M + 127) // 128
        pp_gbs = 8.0 * (5 + nb_blocks) * n_local / (pp_ms * 1e-3) / 1e9 if pp_ms > 0 else None
        per_point = {"bound": "hbm", "ms_per_step": pp_ms, "alg_bytes_per_point": 8.0 * (5 + nb_blocks), "achieved": pp_gbs, "peak": hbm_peak, "unit": "GB/s",
                     "frac": pp_gbs / hbm_peak if pp_gbs else None,
                     "note": "two ~10 us launches per 151 552-point chunk (perpoint + fixed-order scalar reduce): launch-latency-bound, 0.1 % of the step; "
                             "the same kernel given one 1e7-point launch moves 5.0 TB/s (profiles/r02f_perpoint_standalone.jsonl)"}
        metric = METRIC
        if f32:
            metric = METRIC.replace("FP64", "Float32 fast mode: 3xTF32 tcgen05 stages, FP64 solve / reductions")
        if emu:
            metric = METRIC.replace("FP64", "FP64 with S6 emulated FP64-accurately on the INT8 tensor path")
        line = {"metric": metric, "value": value, "unit": UNIT,
                "n_gpus": world, "steps": args.steps, "warmup": n_warm, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": args.dtype,
                "data": "synthetic" + (" (generated on the device)" if on_device else ""),
                "config": svgp_config(w, N_total, world, n_local),
                "elbo": val, "gpu_launches": launches, "clocks": clk, "roofline": roof, "per_point_stage": per_point, "kernels": kernels}
        if e2e:
            line["e2e"] = e2e
        if correctness:
            line["correctness"] = correctness
        if world == 1 and not args.no_cpu_baseline:
            cores = host_threads()
            n_s = min(65536, n_local)
            if Xh is not None:
                Xs, ys = Xh[:n_s].numpy(), yh[:n_s].numpy()
            elif on_device:  # the resident data set was generated on the device: regenerate the same rows there (block-seeded) and fetch them
                Xs_d, ys_d = gen_rows_device(w, 0, n_s, wvec, dev)
                Xs, ys = Xs_d.cpu().numpy(), ys_d.cpu().numpy()
                del Xs_d, ys_d
            else:
                Xs, ys = gen_rows(w, 0, n_s, wvec)
            pps, times, (ref, rg) = time_oracle(w, Z, m, A, Xs, ys, 3, num_data)
            line["cpu_baseline"] = {"value": pps, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"rows [0,{n_s}) of the same workload, median of 3 runs ({sum(times):.1f} s total), NumPy/SciPy OpenBLAS threads={cores}",
                                    "gflops": pps * flops_per_point(M, D) / 1e9}
            # the oracle's result on that sample doubles as an in-bench parity check of the CUDA path (same rows, same num_data)
            L.check(lib.agp_svgp_elbo_grad(ctx.h, ds.h, 0, n_s, C.byref(pk.p), num_data, n_s, C.byref(out), C.byref(G)))
            errs = {"m": rel_to_max(gb["m"], rg.m), "Lq": rel_to_max(gb["Lq"], rg.Lq), "Z": rel_to_max(gb["Z"], rg.Z),
                    "variance": rel_to_max(gb["variance"], rg.kernel.variance), "inv_lengthscale": rel_to_max(gb["inv_lengthscale"], rg.kernel.inv_lengthscale)}
            line["correctness"] = {"what": f"CUDA path vs the CPU restatement on rows [0,{n_s}) (the cpu_baseline sample)", "elbo_cuda": out.value, "elbo_oracle": ref,
                                   "elbo_rel": abs(out.value - ref) / abs(ref), "grad_rel_to_max": errs, "tol": 1e-4 if f32 else 1e-10,
                                   "ok": bool(abs(out.value - ref) / abs(ref) < (1e-4 if f32 else 1e-10) and max(errs.values()) < (1e-4 if f32 else 1e-10))}
        emit(line)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_laplace(args, w):
    """C3: a step is one approx_lml(LaplaceApproximation(), lfx, y) on the N = 8192 problem (kernel matrix built on the device, Newton loop,
    lml).  The path does not shard (DESIGN.md): with --gpus N every rank runs an independent replica and `value` is the aggregate."""
    torch, dist, rank, world, local = setup_dist(args)
    import agp_b200 as agp

    n = args.n or w["N"]
    X, y = c3_problem(n)
    f = agp.GP(1.0 * agp.with_lengthscale(agp.SqExponentialKernel(), 1.0))
    lfx = agp.LatentGP(f, agp.BernoulliLikelihood(), 1e-8)(X)
    la = agp.LaplaceApproximation(maxiter=100)
    ctx = agp.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local))
    barrier, timed = make_timer(torch, dist, world, stream)
    peak_dmma, peak_dfma, peak_src = measure_fp64_peak(ctx)
    kw = agp.laplace_api._check_laplace_inputs(lfx, y, **la.newton_kwargs)
    res = {}

    def step():
        res["r"] = agp.laplace_api._run(ctx, **kw)

    def step_grad():
        res["g"] = agp.laplace_approx_lml_and_gradient(la, lfx, y, ctx=ctx)

    for _ in range(max(3, args.warmup)):
        step()
    l0 = ctx.launch_count()
    clocks = ClockSampler(local) if rank == 0 else None
    ms = timed(step, args.steps)
    clk = clocks.stop() if clocks else {}
    launches = ctx.launch_count() - l0
    r = res["r"]
    last = snapshot(f_opt=r.f, lml=r.lml, newton_steps=r.steps)
    iters = r.steps + (0 if r.converged else 1)  # a converged loop reuses its last cache for the lml (DESIGN.md section 2)
    it_per_s = world * iters * args.steps / (ms * 1e-3)
    ms_iter = ms / args.steps / iters
    step_grad()
    ms_g = timed(step_grad, max(1, min(args.steps, 3))) / max(1, min(args.steps, 3))
    flop_it = laplace_flops_per_iteration(n)
    achieved = flop_it / (ms_iter * 1e-3) / 1e12
    # yard-stick (not part of any product path): the vendor dense Cholesky (torch.linalg.cholesky_ex -> cuSOLVER potrf) on a matrix of the same size
    yard = None
    if rank == 0:
        try:
            g = torch.Generator(device="cuda").manual_seed(1)
            Bm = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
            Bm = Bm @ Bm.T / n + torch.eye(n, dtype=torch.float64, device="cuda")
            for _ in range(2):
                torch.linalg.cholesky_ex(Bm)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                torch.linalg.cholesky_ex(Bm)
            e1.record()
            torch.cuda.synchronize()
            ms_cus = e0.elapsed_time(e1) / 5
            yard = {"cusolver_potrf_ms": ms_cus, "cusolver_potrf_tflops": n ** 3 / 3 / (ms_cus * 1e-3) / 1e12,
                    "note": "torch.linalg.cholesky_ex (cuSOLVER) on a random SPD matrix of the same size; one Newton iteration is one such factorisation "
                            "(+ the factor's block inverses, which this library's kernel also produces) + 6 n^2 of matrix-vector work"}
            del Bm
        except Exception as e:  # noqa: BLE001
            yard = {"error": str(e)[:200]}
    if rank == 0:
        roof = {"bound": "tensor", "kernel": "blocked Cholesky of B = I + sqrt(W) K sqrt(W) (potrf_trinv128 + DMMA panel / trailing GEMMs) and the Newton update",
                "achieved": achieved, "peak": peak_dmma, "unit": "TFLOP/s", "frac": achieved / peak_dmma, "traffic": None,
                "alg_flop_per_iteration": flop_it, "ms_per_newton_iteration": ms_iter,
                "peak_source": f"FP64 DMMA issue peak {peak_src}; DFMA {peak_dfma and round(peak_dfma, 2)} TFLOP/s"}
        line = {"metric": LAPLACE_METRIC, "value": it_per_s, "unit": LAPLACE_UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": w["label"], "N": n, "D": w["D"], "parallelism": f"replicas x{world} (the path does not shard)",
                           "l2": "K, B and L are 537 MB each: far beyond the 126 MB L2"},
                "lml": r.lml, "newton_steps": r.steps, "newton_iterations_per_step": iters, "gpu_launches": launches, "clocks": clk, "roofline": roof,
                "lml_and_gradient_ms": ms_g, "yardstick": yard,
                "e2e": {"value": it_per_s, "unit": LAPLACE_UNIT, "ms_per_step": ms / args.steps, "h2d_bytes_per_step": 8 * n * (w["D"] + 1) * world,
                        "d2h_bytes_per_step": 8 * (n + 1) * world,
                        "note": "the timed call IS the end-to-end call: host X, y in, host f_opt and lml out, every step (the kernel matrix is built on the device)"}}
        if world == 1 and not args.no_cpu_baseline:
            n_cpu = 2048
            t, steps = time_oracle_laplace(n_cpu, 3)
            gflops = laplace_flops_per_iteration(n_cpu) * (steps + 1) / t / 1e9
            line["cpu_baseline"] = {"value": gflops * 1e9 / flop_it, "unit": LAPLACE_UNIT, "cores": host_threads(), "kind": "port", "gflops": gflops,
                                    "sample": f"the same recipe at n={n_cpu} ({steps + 1} Newton iterations, median of 3: {t:.2f} s), extrapolated to N={n} by n^3/3 + 6 n^2"}
        emit(line)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


C1_METRIC = "SVGP ELBO+grad minibatch evaluations/sec (batch 100, FP64)"
C1_UNIT = "evaluations/s"


def c1_problem(M: int):
    """examples/a-regression/script.jl:31-35, :62-69, :89-90, :145-146 with the SURVEY.md section 8(d) seed."""
    rng = np.random.default_rng(1234)
    N = 10_000
    x = rng.uniform(-1, 1, N)
    y = np.sin(3 * np.pi * x) + 0.3 * np.cos(9 * np.pi * x) + 0.5 * np.sin(7 * np.pi * x) + 0.3 * rng.normal(size=N)
    return x, y, x[:M].copy()


def time_oracle_c1(M: int, n_eval: int):
    from threadpoolctl import threadpool_limits

    from oracle import kernels as ok, likelihoods as ol, svgp as osv

    x, y, z = c1_problem(M)
    s_or = osv.SVGP(ok.Kernel("se", 1.3, np.array([1 / 0.3])), z, np.zeros(M), np.eye(M), jitter=1e-5)
    lik = ol.Likelihood("gaussian", 0.3)
    with threadpool_limits(limits=host_threads()):
        for w in range(5):
            osv.elbo_and_grad(s_or, x[:100], y[:100], lik, ol.Expectation(), num_data=1e4)
        t0 = time.perf_counter()
        for i in range(n_eval):
            lo = 100 * (i % 100)
            osv.elbo_and_grad(s_or, x[lo:lo + 100], y[lo:lo + 100], lik, ol.Expectation(), num_data=1e4)
        return n_eval / (time.perf_counter() - t0)


def run_reference_c1(args, w):
    cores = host_threads()
    n_eval = 100 * max(1, args.steps)
    for _ in range(min(1, args.warmup)):
        time_oracle_c1(w["M"], 100)
    value = time_oracle_c1(w["M"], n_eval)
    line = {"impl": "reference", "metric": C1_METRIC, "value": value, "unit": C1_UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * 100 / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": w["label"], "N": w["N"], "M": w["M"], "D": 1, "parallelism": f"replicas x{args.gpus} (a 100-point minibatch does not shard)"},
            "cpu_baseline": {"value": value, "unit": C1_UNIT, "cores": cores, "kind": "port", "sample": f"{n_eval} minibatch evaluations (M={w['M']}), NumPy/SciPy OpenBLAS threads={cores}"},
            "e2e": {"value": value, "unit": C1_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference-algorithm CPU restatement (oracle/, NumPy + OpenBLAS); Julia is not installed so ApproximateGPs.jl itself cannot run"}
    print(json.dumps(line), flush=True)


def run_c1(args, w):
    """C1: every evaluation is agp_svgp_stepper_eval on a 100-point view of the resident data set: the flat parameter vector goes in from
    host memory and ELBO + flat gradient come back to host memory on EVERY evaluation (that is what an optimiser step is), so `value` is
    already end to end for the parameters; the e2e leg additionally uploads the minibatch's (x, y) from host memory before each evaluation."""
    torch, dist, rank, world, local = setup_dist(args)
    import agp_b200 as agp
    from agp_b200 import _lib as L

    ctx = agp.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local))
    barrier, timed = make_timer(torch, dist, world, stream)
    lib = ctx.lib
    res = {}
    for M in (w["M"], 50 if w["M"] != 50 else 20):
        x, y, z = c1_problem(M)
        f = agp.GP(1.3 * agp.with_lengthscale(agp.SqExponentialKernel(), 0.3))
        sva = agp.SparseVariationalApproximation(f(z, 1e-5), agp.MvNormal(np.zeros(M), chol_lower=np.eye(M)))
        ds = agp.DeviceData(x, y, ctx=ctx)
        fo = agp.FlatELBO(sva, agp.FiniteGP(f, ds, 0.3), None, num_data=1e4, ctx=ctx)
        xflat = fo.x0.copy()
        g = np.zeros(fo.size)
        out = C.c_double()
        px, pg = L.dptr(xflat), L.dptr(g)

        def epoch():
            for b in range(100):
                L.check(lib.agp_svgp_stepper_eval(fo._stepper, ds.h, 100 * b, 100, px, 1e4, 0, C.byref(out), pg))

        ds_mb = agp.DeviceData(capacity=100, D=1, ctx=ctx)
        xh, yh = np.ascontiguousarray(x[:, None]), np.ascontiguousarray(y)

        def epoch_e2e():
            for b in range(100):
                lo = 100 * b
                L.check(lib.agp_dataset_upload(ds_mb.h, xh[lo:lo + 100].ctypes.data_as(C.c_void_p), 100, 1, L.POINT_MAJOR, yh[lo:lo + 100].ctypes.data_as(C.c_void_p), L.Y_F64, L.HOST))
                L.check(lib.agp_svgp_stepper_eval(fo._stepper, ds_mb.h, 0, 100, px, 1e4, 0, C.byref(out), pg))

        for _ in range(max(3, args.warmup)):
            epoch()
        l0 = ctx.launch_count()
        clocks = ClockSampler(local) if (rank == 0 and M == w["M"]) else None
        ms = timed(epoch, args.steps)
        clk = clocks.stop() if clocks else {}
        launches = ctx.launch_count() - l0
        if M == w["M"]:  # the evaluation `value` is quoted on: the last minibatch of the last timed epoch
            last = snapshot(elbo=out.value, grad_flat=g)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            epoch()
        wall = time.perf_counter() - t0
        epoch_e2e()
        ms_e = timed(epoch_e2e, args.steps)
        # the throughput path on the same evaluations (what round 1 shipped for this configuration)
        fo_big = agp.FlatELBO(sva, agp.FiniteGP(f, ds, 0.3), None, num_data=1e4, ctx=ctx, resident=False)
        fo_big.value_and_gradient(xflat, offset=0, count=100)
        t0 = time.perf_counter()
        for b in range(100):
            fo_big.value_and_gradient(xflat, offset=100 * b, count=100)
        t_big = (time.perf_counter() - t0) / 100
        res[M] = dict(us_per_evaluation=1e3 * ms / args.steps / 100, us_per_evaluation_wall=1e6 * wall / args.steps / 100, us_per_evaluation_e2e=1e3 * ms_e / args.steps / 100,
                      us_per_evaluation_throughput_path=1e6 * t_big, launches_per_evaluation=launches / args.steps / 100, elbo=out.value, clk=clk,
                      small_path_evaluations=fo.path_counts()[0])
        fo.close()
        fo_big.close()
    if rank == 0:
        M = w["M"]
        r = res[M]
        value = world * 1e6 / r["us_per_evaluation"]
        line = {"metric": C1_METRIC, "value": value, "unit": C1_UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": r["us_per_evaluation"] * 100 / 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": w["label"], "N": w["N"], "M": M, "D": 1, "parallelism": f"replicas x{world} (a 100-point minibatch does not shard)",
                           "l2": "latency-bound: the whole working set (~100 KB) is L1 / L2 resident by design"},
                "elbo": r["elbo"], "gpu_launches": int(r["launches_per_evaluation"] * 100 * args.steps), "clocks": r["clk"],
                "us_per_evaluation": {f"M{m}": v for m, v in res.items()},
                "roofline": {"bound": "latency", "kernel": "svgp_small_kernel (one CTA, one launch per evaluation)", "achieved": None, "peak": None, "unit": None, "frac": None,
                             "traffic": None, "note": "one 1024-thread CTA working out of L1: neither HBM nor the FP64 pipe is the bound, launch + synchronisation + "
                                                      "the M sequential pivots of the Cholesky are; the figure of merit is microseconds per evaluation"},
                "e2e": {"value": world * 1e6 / r["us_per_evaluation_e2e"], "unit": C1_UNIT, "ms_per_step": r["us_per_evaluation_e2e"] * 100 / 1e3,
                        "h2d_bytes_per_step": 100 * (8 * 200 + 8 * (4 + 1 + M + M + M * M)), "d2h_bytes_per_step": 100 * 8 * (1 + 4 + 1 + M + M + M * M)}}
        if world == 1 and not args.no_cpu_baseline:
            cpu = {m: time_oracle_c1(m, 300) for m in res}
            line["cpu_baseline"] = {"value": cpu[M], "unit": C1_UNIT, "cores": host_threads(), "kind": "port",
                                    "sample": f"300 minibatch evaluations per M, NumPy/SciPy OpenBLAS threads={host_threads()}",
                                    "us_per_evaluation": {f"M{m}": 1e6 / v for m, v in cpu.items()}}
        emit(line)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--points", "--n", dest="n", type=int, default=0, help="override the number of points (debugging only; the line says so)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip the N > 1 sharded-vs-single-rank correctness evaluation")
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32", "f32_tc_solve", "f64emu"], help="f64emu: Float64 tolerance with S6 as an FP64-accurate INT8-slice product on tcgen05 (AGP_COMPUTE_F64_EMU; its own line, never the headline); f32: the Float32 fast mode (3xTF32 on tcgen05 for the GEMM-shaped sweep stages); "
                                                                             "reported as its own line, never as the Float64 headline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (ELBO and gradients; Laplace: f_opt, lml) as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the b200 arm's outputs")
    w = dict(WORKLOADS[args.workload])
    if args.n:
        w["N"] = args.n
        w["label"] += f" [N overridden to {args.n}]"
    if args.impl == "reference":
        return run_reference(args, w)
    if w.get("laplace"):
        return run_laplace(args, w)
    if w.get("small"):
        return run_c1(args, w)
    return run_svgp(args, w)


if __name__ == "__main__":
    main()
