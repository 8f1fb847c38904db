"""Kernel sums / products (KernelFunctions `k1 + k2`, `k1 * k2`; public through `@reexport using AbstractGPs`, src/ApproximateGPs.jl:5) on the
device path: SVGP ELBO + every gradient, the kernel matrix behind the predictions, and the Laplace objective, against the oracle (whose
reverse pass for these kernels is checked against finite differences in tests/test_oracle_svgp.py)."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from _cases import make_problem, oracle_objects, record_parity, rel_err  # noqa: E402

from oracle import kernels as ok, laplace as olap, likelihoods as ol, svgp as osv  # noqa: E402

pytestmark = pytest.mark.gpu

NAMES = {"se": "SqExponentialKernel", "matern32": "Matern32Kernel", "matern52": "Matern52Kernel"}
COMPS = (("se", 0.7, 1.3), ("matern32", 1.1, 0.6), ("matern52", 0.4, 2.0))


@pytest.fixture(scope="module")
def agp():
    import agp_b200

    return agp_b200


def _device_kernel(agp, op, comps, variance, inv):
    terms = [v * agp.ScaleTransform(getattr(agp, NAMES[kd])(), s) for kd, v, s in comps]
    k = terms[0]
    for t in terms[1:]:
        k = k + t if op == "sum" else k * t
    k = variance * k
    return agp.ScaleTransform(k, inv[0]) if inv.size == 1 else agp.ARDTransform(k, inv)


@pytest.mark.parametrize("op", ["sum", "product"])
@pytest.mark.parametrize("centered,D,M,N,ard", [(False, 3, 40, 700, True), (True, 1, 24, 300, False), (False, 8, 200, 1500, False)])
# (the Centered case uses a Gaussian likelihood, inducing points drawn independently of the data and a short length scale: with the default
#  D = 1 problem Kuu has a condition number of 1e9 and the un-whitened random q gives marginal variances whose Poisson expectation is 1e14)
def test_svgp_sum_product(agp, op, centered, D, M, N, ard):
    p = make_problem(seed=21, kind="se", N=N, M=M, D=D, lik="gaussian" if centered else "poisson_exp", centered=centered, ard=ard, lengthscale=1.0 if D == 8 else (0.15 if D == 1 else None),
                     zdist="data" if D != 1 else "random")
    comps = COMPS if D != 8 else COMPS[:2]
    _, lik, ex = oracle_objects(p)
    s = osv.SVGP(ok.Kernel(op, p["variance"], p["inv"], 0.0, comps), p["Z"], p["m"], p["A"], jitter=1e-6, centered=centered)
    ref, rg = osv.elbo_and_grad(s, p["X"], p["y"], lik, ex, num_data=5 * N)
    f = agp.GP(_device_kernel(agp, op, comps, p["variance"], p["inv"]))
    sva = agp.SparseVariationalApproximation(agp.Centered() if centered else agp.NonCentered(), f(p["Z"], 1e-6), agp.MvNormal(p["m"], chol_lower=p["A"]))
    lfx = agp.LatentGP(f, agp.GaussianLikelihood(p["sigma2"]) if centered else agp.PoissonLikelihood(), 1e-18)(p["X"])
    val, g = agp.elbo_and_gradient(sva, lfx, p["y"], num_data=5 * N)
    errs = dict(elbo=abs(val - ref) / abs(ref), m=rel_err(g.m, rg.m), Lq=rel_err(g.Lq, rg.Lq), Z=rel_err(g.Z, rg.Z), variance=rel_err(g.variance, rg.kernel.variance),
                inv_lengthscale=rel_err(g.inv_lengthscale, rg.kernel.inv_lengthscale), comp_variance=rel_err(g.comp_variance, rg.kernel.comp_variance),
                comp_inv_lengthscale=rel_err(g.comp_inv_lengthscale, rg.kernel.comp_inv_lengthscale))
    label = f"kernel {op} of {len(comps)} D={D} M={M} N={N} cent={centered}"
    print(f"\n[{label}] elbo={val:.10f} " + " ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    # named exception (the same one as in test_gpu_svgp.py): Centered + SqExponential components, cond(Kuu) ~ 1e5 -- two backward-stable
    # float64 evaluations differ by cond * eps; measured 1.2e-11 .. 1.1e-10 on d/dvariance across builds that only reorder the sums
    # inside the 32 x 32 Cholesky blocks
    tol = 1e-9 if centered else 1e-10
    record_parity(label, errs, tol=tol)
    for k, v in errs.items():
        assert v < tol, (k, v)
    # the flat-vector interface carries the component parameters behind Lq
    fo = agp.FlatELBO(sva, lfx, p["y"], num_data=5 * N)
    v2, g2 = fo.value_and_gradient(fo.x0)
    u = fo.unflatten(g2)
    assert abs(v2 - val) <= 1e-12 * abs(val)
    assert np.allclose(u["comp_variance"], g.comp_variance, rtol=1e-12, atol=0) and np.allclose(u["comp_inv_lengthscale"], g.comp_inv_lengthscale, rtol=1e-12, atol=0)
    assert fo.path_counts()[0] == 0  # sums / products take the throughput path
    fo.close()


def test_kernelmatrix_and_prediction(agp):
    rng = np.random.default_rng(3)
    X, Y = rng.normal(size=(150, 3)), rng.normal(size=(70, 3))
    inv = np.array([0.9, 1.1, 0.7])
    for op in ("sum", "product"):
        k = ok.Kernel(op, 1.7, inv, 0.0, COMPS)
        kd = _device_kernel(agp, op, COMPS, 1.7, inv)
        assert rel_err(agp.kernelmatrix(kd, X, Y), ok.kernelmatrix(k, X, Y)) < 1e-13
        K1 = agp.kernelmatrix(kd, X)
        assert rel_err(K1, ok.kernelmatrix(k, X)) < 1e-13 and np.array_equal(K1, K1.T)
        # posterior marginals of an SVGP with this kernel
        p = make_problem(seed=5, kind="se", N=150, M=30, D=3, lik="gaussian")
        s = osv.SVGP(k, p["Z"], p["m"], p["A"], jitter=1e-6)
        f = agp.GP(kd)
        sva = agp.SparseVariationalApproximation(f(p["Z"], 1e-6), agp.MvNormal(p["m"], chol_lower=p["A"]))
        mu, var = agp.mean_and_var(agp.posterior(sva), Y)
        rmu, rvar = osv.mean_and_var(s, Y)
        assert rel_err(mu, rmu) < 1e-10 and rel_err(var, rvar) < 1e-10


@pytest.mark.parametrize("op", ["sum", "product", "se_ard", "linear"])
def test_laplace_sum_product(agp, op):
    # (se_ard / linear, at D = 3: the per-dimension inverse lengthscales and LinearKernel's offset in the Laplace kernel gradient)
    X, y = olap.generate_data()
    rng = np.random.default_rng(17)
    Xn = np.linspace(-1.0, 8.0, 37)
    if op in ("sum", "product"):
        comps = (("se", 1.5, 0.8), ("matern52", 0.6, 2.5))
        k = ok.Kernel(op, 2.0, np.array([1.2]), 0.0, comps)
        kd = _device_kernel(agp, op, comps, 2.0, np.array([1.2]))
    else:
        X = np.column_stack([X, rng.uniform(0.0, 4.0, size=(len(y), 2))])
        Xn = rng.uniform(-1.0, 5.0, size=(37, 3))
        if op == "se_ard":
            inv = np.array([1.2, 0.7, 1.6])
            k, kd = ok.Kernel(ok.SE, 2.0, inv), 2.0 * agp.ARDTransform(agp.SqExponentialKernel(), inv)
        else:
            k, kd = ok.Kernel(ok.LINEAR, 0.5, np.array([0.8]), 0.3), 0.5 * agp.ScaleTransform(agp.LinearKernel(0.3), 0.8)
    lik = ol.Likelihood(ol.BERNOULLI_LOGIT)
    K = ok.kernelmatrix(k, X) + 1e-8 * np.eye(len(y))
    lml, K_bar, f_opt, steps = olap.lml_and_grad_K(lik, y, K)
    dX, _, kg = ok.kernelmatrix_pullback(k, X, None, K_bar)
    f = agp.GP(kd)
    lfx = agp.LatentGP(f, agp.BernoulliLikelihood(), 1e-8)(X)
    r = agp.laplace_approx_lml_and_gradient(agp.LaplaceApproximation(), lfx, y)
    errs = dict(lml=abs(r.lml - lml) / abs(lml), variance=rel_err(r.grad.variance, kg.variance), inv_lengthscale=rel_err(r.grad.inv_lengthscale, kg.inv_lengthscale),
                X=rel_err(r.grad.X, dX))
    if op in ("sum", "product"):
        errs.update(comp_variance=rel_err(r.grad.comp_variance, kg.comp_variance), comp_inv_lengthscale=rel_err(r.grad.comp_inv_lengthscale, kg.comp_inv_lengthscale))
    if op == "linear":
        errs.update(linear_c=rel_err(r.grad.linear_c, kg.c))
    print(f"\n[laplace kernel {op}] lml={r.lml:.12f} " + " ".join(f"{k_}={v:.1e}" for k_, v in errs.items()))
    record_parity(f"laplace kernel {op}", errs, tol=1e-8)
    assert errs["lml"] < 1e-10 and r.steps == steps
    assert np.shape(r.grad.inv_lengthscale) == np.shape(k.inv_lengthscale)
    for k_, v in errs.items():
        assert v < 1e-8, (k_, v)
    # prediction through the cache
    post = agp.posterior(agp.LaplaceApproximation(), lfx, y)
    mu, var = agp.mean_and_var(post, Xn)
    cache = olap.train_intermediates(lik, y, K, f_opt)
    rmu, rvar = olap.predict_mean_and_var(k, X, cache, Xn)
    assert rel_err(mu, rmu) < 1e-9 and rel_err(var, rvar) < 1e-8
