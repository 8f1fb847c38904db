"""CPU: the parts of bench.py that run without a GPU -- synthetic data generation, and the `--impl reference` arm (the CPU
restatement timed on the host cores), whose JSON line must carry the contract's keys."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_synthetic_rows_are_independent_of_the_slice():
    import bench

    w = dict(bench.WORKLOADS["c4"])
    wvec, Z, m, A = bench.make_params(w)
    Xa, ya = bench.gen_rows(w, 0, 3000, wvec)
    Xb, yb = bench.gen_rows(w, 1000, 2000, wvec)
    assert np.array_equal(Xa[1000:2000], Xb) and np.array_equal(ya[1000:2000], yb)
    lo = bench.BLOCK - 5  # a slice that straddles a generation block
    Xc, yc = bench.gen_rows(w, lo, lo + 10, wvec)
    Xd, _ = bench.gen_rows(w, lo + 5, lo + 6, wvec)
    assert np.array_equal(Xc[5:6], Xd) and Xc.shape == (10, 8) and np.all(yc >= 0)
    assert Z.shape == (1024, 8) and np.all(np.diag(A) > 0) and np.allclose(A, np.tril(A))
    assert bench.flops_per_point(1024, 8) == 6 * 1024 * 1024 + 6 * 1024 * 8
    assert abs(sum(bench.class_flops_per_point(1024, 8).values()) + bench.SAVED_BY_ALGEBRA(1024, 8) - bench.flops_per_point(1024, 8)) < 1e-6


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, OPENBLAS_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "points/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"] and d["dtype"] == "f64" and d["data"] == "synthetic"


def test_argument_errors():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and "error" in out.stderr, out.stderr[-2000:]


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_step_results(tmp_path):
    """--dump-outputs writes the ELBO and every gradient buffer of the last timed step; on the flagship workload cut to its first
    16384 rows they match the CPU restatement on the same rows."""
    import bench
    from oracle import svgp as osv

    n = 16384
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--points", str(n), "--steps", "2", "--warmup", "1", "--no-e2e",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2
    got = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert set(got) == {"elbo", "grad_m", "grad_Lq", "grad_Z", "grad_variance", "grad_inv_lengthscale", "grad_lik_sigma2"}
    assert all(a.dtype == np.float64 for a in got.values())
    assert abs(got["elbo"][0] - d["elbo"]) <= 1e-12 * abs(d["elbo"])
    w = dict(bench.WORKLOADS["c4"], N=n)
    wvec, Z, m, A = bench.make_params(w)
    X, y = bench.gen_rows(w, 0, n, wvec)
    s, lik, ex = bench.oracle_objects(w, Z, m, A)
    ref, rg = osv.elbo_and_grad(s, X, y, lik, ex, num_data=float(n))
    assert abs(got["elbo"][0] - ref) < 1e-10 * abs(ref)
    for k, r in (("m", rg.m), ("Lq", rg.Lq), ("Z", rg.Z), ("variance", rg.kernel.variance), ("inv_lengthscale", rg.kernel.inv_lengthscale)):
        assert got["grad_" + k].shape == np.shape(np.atleast_1d(r)) and bench.rel_to_max(got["grad_" + k], r) < 1e-10, k
