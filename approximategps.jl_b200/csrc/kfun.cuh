// kfun.cuh -- covariance functions and likelihood expectations evaluated on the device.
//
// Semantics follow what the reference reaches through KernelFunctions / Distances
// (cov(f.prior, z, x), SVA.jl:216) and GPLikelihoods.expected_loglikelihood (SVA.jl:355); see
// oracle/kernels.py and oracle/likelihoods.py for the CPU restatement these are tested against.
#pragma once
#include <math.h>
#include "../../include/agp.h"
#include "common.cuh"

namespace agp {

constexpr int MAXD = AGP_MAX_D;  // compile-time bound on the input dimension handled on device (include/agp.h)
constexpr int MAXC = AGP_MAX_COMPONENTS;

struct KernelParams {
  int kind;
  int D;
  int M;  // valid inducing points (rows >= M of every padded operand are zero)
  int ard;
  double variance;
  double c;
  double s[MAXD];  // per-dimension input scale (ScaleTransform replicated, or ARDTransform)
  // kind == AGP_KERNEL_SUM / AGP_KERNEL_PRODUCT: k = variance * F(u), F(u) = sum_c / prod_c  cv[c] kappa_{ckind[c]}(ca[c] u) with u the
  // squared distance of the inputs scaled by s[] and ca[c] = (component inverse lengthscale)^2; f0 = F(0) (1 for the plain kinds)
  int ncomp;
  int ckind[MAXC];
  double cv[MAXC];
  double ca[MAXC];
  double f0;
};
__host__ __device__ __forceinline__ bool kernel_is_composite(int kind) { return kind == AGP_KERNEL_SUM || kind == AGP_KERNEL_PRODUCT; }

// Padded row width of the operands of the Kuf generator: Dq = D rounded up to 4 (one DMMA k-step); a padded row is
// [v_0 .. v_{D-1}, 0.., |v|^2, 0] with Dq + 2 doubles (16-byte aligned rows).
__host__ __device__ __forceinline__ int kuf_dp(int D) { return (D + 3) & ~3; }

// kappa(u): u = squared distance of the scaled inputs (stationary) or their dot product (linear)
__device__ __forceinline__ double kappa(int kind, double u, double c) {
  if (kind == AGP_KERNEL_SE) return exp(-0.5 * u);
  if (kind == AGP_KERNEL_LINEAR) return u + c;
  const double d = sqrt(u);
  if (kind == AGP_KERNEL_MATERN32) {
    const double r = 1.7320508075688772 * d;
    return (1.0 + r) * exp(-r);
  }
  const double r = 2.23606797749979 * d;
  return (1.0 + r + (5.0 / 3.0) * u) * exp(-r);
}
// kappa and d kappa / d u in one go (finite at u == 0)
__device__ __forceinline__ void kappa_and_du(int kind, double u, double c, double& k, double& dk) {
  if (kind == AGP_KERNEL_SE) {
    k = exp(-0.5 * u);
    dk = -0.5 * k;
    return;
  }
  if (kind == AGP_KERNEL_LINEAR) {
    k = u + c;
    dk = 1.0;
    return;
  }
  const double d = sqrt(u);
  if (kind == AGP_KERNEL_MATERN32) {
    const double r = 1.7320508075688772 * d;
    const double e = exp(-r);
    k = (1.0 + r) * e;
    dk = -1.5 * e;
    return;
  }
  const double r = 2.23606797749979 * d;
  const double e = exp(-r);
  k = (1.0 + r + (5.0 / 3.0) * u) * e;
  dk = -(5.0 / 6.0) * (1.0 + r) * e;
}
// exp(x) for x <= 0 (the stationary covariance functions only ever need a decaying exponential): table-driven,
//   x = (64 q + j) ln2/64 + r,  |r| <= ln2/128,  exp(x) = 2^q T[j] (1 + p(r)),  p = degree-6 Taylor of expm1 (|r|^7/5040 < 3e-20)
// 13 FP64-pipe instructions against ~25 of the CUDA library routine (which spends the rest on the x > 0 / overflow paths this
// caller cannot reach).  Used by kuf_gen_kernel, which is bound by the FP64 pipe (8 FMAs of distance + the exponential per element),
// not by HBM.  Error against mpmath over [-708, 0]: below 1 ulp (exact emulation of this
// operation sequence, and tests/test_gpu_svgp.py::test_kernel_function_values on the device).  x < -708 (result < 1e-307) returns 0.
__device__ const double c_exp2_tab[64] = {
    0x1.0000000000000p+0, 0x1.02c9a3e778061p+0, 0x1.059b0d3158574p+0, 0x1.0874518759bc8p+0,
    0x1.0b5586cf9890fp+0, 0x1.0e3ec32d3d1a2p+0, 0x1.11301d0125b51p+0, 0x1.1429aaea92de0p+0,
    0x1.172b83c7d517bp+0, 0x1.1a35beb6fcb75p+0, 0x1.1d4873168b9aap+0, 0x1.2063b88628cd6p+0,
    0x1.2387a6e756238p+0, 0x1.26b4565e27cddp+0, 0x1.29e9df51fdee1p+0, 0x1.2d285a6e4030bp+0,
    0x1.306fe0a31b715p+0, 0x1.33c08b26416ffp+0, 0x1.371a7373aa9cbp+0, 0x1.3a7db34e59ff7p+0,
    0x1.3dea64c123422p+0, 0x1.4160a21f72e2ap+0, 0x1.44e086061892dp+0, 0x1.486a2b5c13cd0p+0,
    0x1.4bfdad5362a27p+0, 0x1.4f9b2769d2ca7p+0, 0x1.5342b569d4f82p+0, 0x1.56f4736b527dap+0,
    0x1.5ab07dd485429p+0, 0x1.5e76f15ad2148p+0, 0x1.6247eb03a5585p+0, 0x1.6623882552225p+0,
    0x1.6a09e667f3bcdp+0, 0x1.6dfb23c651a2fp+0, 0x1.71f75e8ec5f74p+0, 0x1.75feb564267c9p+0,
    0x1.7a11473eb0187p+0, 0x1.7e2f336cf4e62p+0, 0x1.82589994cce13p+0, 0x1.868d99b4492edp+0,
    0x1.8ace5422aa0dbp+0, 0x1.8f1ae99157736p+0, 0x1.93737b0cdc5e5p+0, 0x1.97d829fde4e50p+0,
    0x1.9c49182a3f090p+0, 0x1.a0c667b5de565p+0, 0x1.a5503b23e255dp+0, 0x1.a9e6b5579fdbfp+0,
    0x1.ae89f995ad3adp+0, 0x1.b33a2b84f15fbp+0, 0x1.b7f76f2fb5e47p+0, 0x1.bcc1e904bc1d2p+0,
    0x1.c199bdd85529cp+0, 0x1.c67f12e57d14bp+0, 0x1.cb720dcef9069p+0, 0x1.d072d4a07897cp+0,
    0x1.d5818dcfba487p+0, 0x1.da9e603db3285p+0, 0x1.dfc97337b9b5fp+0, 0x1.e502ee78b3ff6p+0,
    0x1.ea4afa2a490dap+0, 0x1.efa1bee615a27p+0, 0x1.f50765b6e4540p+0, 0x1.fa7c1819e90d8p+0};
__device__ __forceinline__ double exp_nonpos(double x) {
  const double t = fma(x, 0x1.71547652b82fep+6, 0x1.8p52);  // low mantissa bits of t = k = round(64 x / ln2) (two's complement)
  const double kd = t - 0x1.8p52;
  double r = fma(-kd, 0x1.62e42fef00000p-7, x);  // exact: the high part of ln2/64 has 20 trailing zero bits, |k| < 2^17
  r = fma(-kd, 0x1.473de6af278edp-40, r);
  const int ki = __double2loint(t);
  const double tj = __ldg(c_exp2_tab + (ki & 63));
  double p = fma(r, 1.0 / 720.0, 1.0 / 120.0);
  p = fma(p, r, 1.0 / 24.0);
  p = fma(p, r, 1.0 / 6.0);
  p = fma(p, r, 0.5);
  p = fma(p * r, r, r);  // expm1(r)
  const double v = fma(tj, p, tj);
  const double res = __hiloint2double(__double2hiint(v) + ((ki >> 6) << 20), __double2loint(v));
  return x < -708.0 ? 0.0 : res;
}


// kappa (and d kappa / d u) with the table-driven exponential: the stand-alone Kuf generator of S1
__device__ __forceinline__ void kappa_and_du_gen(int kind, double u, double c, double& k, double& dk) {
  if (kind == AGP_KERNEL_SE) {
    k = exp_nonpos(-0.5 * u);
    dk = -0.5 * k;
    return;
  }
  if (kind == AGP_KERNEL_LINEAR) {
    k = u + c;
    dk = 1.0;
    return;
  }
  const double d = sqrt(u);
  if (kind == AGP_KERNEL_MATERN32) {
    const double r = 1.7320508075688772 * d;
    const double e = exp_nonpos(-r);
    k = (1.0 + r) * e;
    dk = -1.5 * e;
    return;
  }
  const double r = 2.23606797749979 * d;
  const double e = exp_nonpos(-r);
  k = (1.0 + r + (5.0 / 3.0) * u) * e;
  dk = -(5.0 / 6.0) * (1.0 + r) * e;
}
// combine |xs|^2, |zs|^2 and xs.zs into u (Distances.jl: GEMM form with max(., 0) for D > 1)
__device__ __forceinline__ double u_from_dot(int kind, double xn, double zn, double dot) {
  if (kind == AGP_KERNEL_LINEAR) return dot;
  return fmax(xn + zn - 2.0 * dot, 0.0);
}

// kappa for every kind, including sums / products of stationary components
__device__ __forceinline__ double kappa_kp(const KernelParams& kp, double u) {
  if (!kernel_is_composite(kp.kind)) return kappa(kp.kind, u, kp.c);
  const bool sum = kp.kind == AGP_KERNEL_SUM;
  double f = sum ? 0.0 : 1.0;
  for (int c = 0; c < kp.ncomp; c++) {
    const double kc = kp.cv[c] * kappa(kp.ckind[c], kp.ca[c] * u, 0.0);
    f = sum ? f + kc : f * kc;
  }
  return f;
}
// F(u), dF/du and, per component, pc[c] = dF/d cv[c], qc[c] = dF/d ca[c]  (products: without divisions, so that a factor that
// underflows to zero gives zeros, not NaNs)
__device__ __forceinline__ void kappa_comp(const KernelParams& kp, double u, double& F, double& dF, double (&pc)[MAXC], double (&qc)[MAXC]) {
  double kc[MAXC], dkc[MAXC];
#pragma unroll
  for (int c = 0; c < MAXC; c++) {
    kc[c] = 1.0;
    dkc[c] = 0.0;
    if (c < kp.ncomp) kappa_and_du(kp.ckind[c], kp.ca[c] * u, 0.0, kc[c], dkc[c]);
  }
  F = dF = 0.0;
  if (kp.kind == AGP_KERNEL_SUM) {
#pragma unroll
    for (int c = 0; c < MAXC; c++) {
      pc[c] = qc[c] = 0.0;
      if (c < kp.ncomp) {
        F = fma(kp.cv[c], kc[c], F);
        dF = fma(kp.cv[c] * kp.ca[c], dkc[c], dF);
        pc[c] = kc[c];
        qc[c] = kp.cv[c] * u * dkc[c];
      }
    }
  } else {
    double tot = 1.0;
#pragma unroll
    for (int c = 0; c < MAXC; c++)
      if (c < kp.ncomp) tot *= kp.cv[c] * kc[c];
    F = tot;
#pragma unroll
    for (int c = 0; c < MAXC; c++) {
      pc[c] = qc[c] = 0.0;
      if (c < kp.ncomp) {
        double oth = 1.0;  // product of the other factors
#pragma unroll
        for (int e = 0; e < MAXC; e++)
          if (e < kp.ncomp && e != c) oth *= kp.cv[e] * kc[e];
        pc[c] = oth * kc[c];
        qc[c] = oth * kp.cv[c] * u * dkc[c];
        dF = fma(oth * kp.cv[c] * kp.ca[c], dkc[c], dF);
      }
    }
  }
}

// ---- likelihood expectations ------------------------------------------------------------------
struct LikParams {
  int kind;
  int method;  // resolved: AGP_EXPECT_ANALYTIC, AGP_EXPECT_GAUSS_HERMITE or AGP_EXPECT_MONTE_CARLO
  int ngh;     // Gauss-Hermite nodes / Monte-Carlo samples per point
  double sigma2;
  unsigned long long seed;  // Monte Carlo
  const double* gh;         // Gauss-Hermite: device buffer owned by the context, nodes at [0, ngh), weights at [AGP_MAX_GH_POINTS, ..)
};

// ---- counter-based normal variates (Philox4x32-10 + Box-Muller) --------------------------------------------------
// eps(seed, point, sample): counter = (point_lo, point_hi, sample, 0), key = (seed_lo, seed_hi); the first two output words
// give u1 in (0, 1], the last two u2 in [0, 1); eps = sqrt(-2 ln u1) cos(2 pi u2).  oracle/likelihoods.py restates it.
__host__ __device__ __forceinline__ void philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1, unsigned (&out)[4]) {
  for (int r = 0; r < 10; r++) {
    const unsigned long long p0 = 0xD2511F53ull * c0, p1 = 0xCD9E8D57ull * c2;
    const unsigned n0 = (unsigned)(p1 >> 32) ^ c1 ^ k0, n1 = (unsigned)p1, n2 = (unsigned)(p0 >> 32) ^ c3 ^ k1, n3 = (unsigned)p0;
    c0 = n0;
    c1 = n1;
    c2 = n2;
    c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0;
  out[1] = c1;
  out[2] = c2;
  out[3] = c3;
}
__device__ __forceinline__ double philox_normal(unsigned long long seed, long long point, int sample) {
  unsigned r[4];
  philox4x32_10((unsigned)point, (unsigned)((unsigned long long)point >> 32), (unsigned)sample, 0u, (unsigned)seed, (unsigned)(seed >> 32), r);
  const unsigned long long a = ((unsigned long long)r[0] << 32) | r[1], b = ((unsigned long long)r[2] << 32) | r[3];
  const double u1 = ((double)(a >> 11) + 1.0) * (1.0 / 9007199254740992.0);  // (0, 1]
  const double u2 = (double)(b >> 11) * (1.0 / 9007199254740992.0);          // [0, 1)
  return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

// (The Gauss-Hermite table lives in a per-context device buffer, LikParams::gh: a device-global __constant__ symbol would be
// shared -- and overwritten mid-kernel -- by every context of the device.)

__device__ __forceinline__ double softplus(double x) { return fmax(x, 0.0) + log1p(exp(-fabs(x))); }
__device__ __forceinline__ double logistic(double x) {
  if (x >= 0.0) return 1.0 / (1.0 + exp(-x));
  const double e = exp(x);
  return e / (1.0 + e);
}

// log Phi(z) and r(z) = phi(z) / Phi(z) for the probit link, overflow-free through erfcx: Phi(z) = erfc(t) / 2 with
// t = -z / sqrt2, r = sqrt(2/pi) / erfcx(t).  (An intentional divergence like the logistic one above: the reference evaluates
// log(normcdf(f)) / log(1 - normcdf(f)), which loses its digits once normcdf(f) rounds to 0 or 1.)
__device__ __forceinline__ void log_ndtr_and_ratio(double z, double& lp, double& r) {
  const double t = -0.7071067811865476 * z;
  const double ex = erfcx(t);
  r = 0.7978845608028654 / ex;
  lp = (t > 0.0) ? log(0.5 * ex) - t * t : log1p(-0.5 * erfc(-t));
}

// digamma(x), x > 0: recurrence up to x >= 10, then the asymptotic series (error < 1e-15)
__device__ __forceinline__ double digamma(double x) {
  double r = 0.0;
  while (x < 10.0) {
    r -= 1.0 / x;
    x += 1.0;
  }
  const double i = 1.0 / x, i2 = i * i;
  const double ser = i2 * (1.0 / 12.0 - i2 * (1.0 / 120.0 - i2 * (1.0 / 252.0 - i2 * (1.0 / 240.0 - i2 * (1.0 / 132.0 - i2 * (691.0 / 32760.0))))));
  return r + log(x) - 0.5 * i - ser;
}

// the part of log p(y | f) that does not depend on f
__device__ __forceinline__ double loglik_const(const LikParams& lp, double y) {
  if (lp.kind == AGP_LIK_POISSON_EXP) return -lgamma(y + 1.0);
  if (lp.kind == AGP_LIK_GAMMA_EXP) return (lp.sigma2 - 1.0) * log(y) - lgamma(lp.sigma2);
  if (lp.kind == AGP_LIK_GAUSSIAN) return -0.5 * (1.8378770664093453 + log(lp.sigma2));
  return 0.0;
}

// log p(y | f), d/df and d/d(likelihood parameter) (closed forms of Distributions.logpdf; the Bernoulli form is the
// overflow-free -softplus(-+f), an intentional divergence from the reference's log(logistic(f)) which returns -Inf for
// |f| > 36.7, SURVEY.md section 7.2).  cst = loglik_const(lp, y).
__device__ __forceinline__ void loglik_d1(const LikParams& lp, double f, double y, double cst, double& ll, double& dll, double& dpar) {
  dpar = 0.0;
  if (lp.kind == AGP_LIK_BERNOULLI_LOGIT) {
    const bool one = y > 0.5;
    ll = -softplus(one ? -f : f);
    dll = (one ? 1.0 : 0.0) - logistic(f);
  } else if (lp.kind == AGP_LIK_BERNOULLI_PROBIT) {  // log Phi(s f), s = +-1
    const double sg = (y > 0.5) ? 1.0 : -1.0;
    double r;
    log_ndtr_and_ratio(sg * f, ll, r);
    dll = sg * r;
  } else if (lp.kind == AGP_LIK_POISSON_EXP) {
    const double lam = exp(f);
    ll = y * f - lam + cst;
    dll = y - lam;
  } else if (lp.kind == AGP_LIK_EXPONENTIAL_EXP) {  // Exponential(scale = exp(f)): -f - y exp(-f)
    const double t = y * exp(-f);
    ll = -f - t;
    dll = -1.0 + t;
  } else if (lp.kind == AGP_LIK_GAMMA_EXP) {  // Gamma(alpha, scale = exp(f)): (alpha-1) log y - y exp(-f) - alpha f - lgamma(alpha)
    const double t = y * exp(-f);
    ll = cst - t - lp.sigma2 * f;
    dll = -lp.sigma2 + t;
    dpar = -f;  // + log y - digamma(alpha), added once per point by the caller
  } else {
    const double r = y - f;
    ll = cst - 0.5 * r * r / lp.sigma2;
    dll = r / lp.sigma2;
    dpar = -0.5 / lp.sigma2 + 0.5 * r * r / (lp.sigma2 * lp.sigma2);
  }
}

// E = E_{N(mu, var)}[log p(y|f)], dE/dmu, dE/dvar, dE/dsigma2 (derivatives of the finite
// quadrature sum, which is what Zygote differentiates in the reference).
__device__ __forceinline__ void expected_loglik(const LikParams& lp, double mu, double var, double y, double& E,
                                                double& dmu, double& dvar, double& ds2, long long point = 0) {
  const double sd = sqrt(var);
  ds2 = 0.0;
  if (lp.method == AGP_EXPECT_MONTE_CARLO) {
    // GPLikelihoods.MonteCarloExpectation(n): mean over n reparameterised samples f = mu + sd * eps of log p(y | f); the
    // derivatives are those of this finite sum (what Zygote differentiates), eps held fixed.
    const double cst = loglik_const(lp, y);
    const double par0 = (lp.kind == AGP_LIK_GAMMA_EXP) ? log(y) - digamma(lp.sigma2) : 0.0;
    double sE = 0.0, sM = 0.0, sS = 0.0, sG = 0.0;
    for (int k = 0; k < lp.ngh; k++) {
      const double eps = philox_normal(lp.seed, point, k);
      const double f = fma(sd, eps, mu);
      double ll, dll, dpar;
      loglik_d1(lp, f, y, cst, ll, dll, dpar);
      sE += ll;
      sM += dll;
      sS = fma(dll, eps, sS);
      sG += dpar;
    }
    const double inv = 1.0 / (double)lp.ngh;
    E = sE * inv;
    dmu = sM * inv;
    dvar = sS * inv / (2.0 * sd);
    ds2 = sG * inv + par0;
    return;
  }
  if (lp.method == AGP_EXPECT_ANALYTIC) {
    const double v = sd * sd;  // Normal(mu, sqrt(var)) re-squared, as in the reference
    if (lp.kind == AGP_LIK_GAUSSIAN) {
      const double r = y - mu, s2 = lp.sigma2;
      E = -0.5 * (1.8378770664093453 + log(s2) + (r * r + v) / s2);
      dmu = r / s2;
      dvar = -0.5 / s2;
      ds2 = -0.5 / s2 + 0.5 * (r * r + v) / (s2 * s2);
    } else if (lp.kind == AGP_LIK_POISSON_EXP) {
      const double e = exp(mu + 0.5 * v);
      E = y * mu - e - lgamma(y + 1.0);
      dmu = y - e;
      dvar = -0.5 * e;
    } else {  // Exponential / Gamma with exp link: E[exp(-f)] = exp(-mu + v/2)
      const double alpha = (lp.kind == AGP_LIK_GAMMA_EXP) ? lp.sigma2 : 1.0;
      const double t = y * exp(-mu + 0.5 * v);
      E = loglik_const(lp, y) - t - alpha * mu;
      dmu = -alpha + t;
      dvar = -0.5 * t;
      if (lp.kind == AGP_LIK_GAMMA_EXP) ds2 = log(y) - digamma(alpha) - mu;
    }
    return;
  }
  const double cst = loglik_const(lp, y);
  const double sq2sd = 1.4142135623730951 * sd;
  double sE = 0.0, sM = 0.0, sS = 0.0, sG = 0.0;
  for (int k = 0; k < lp.ngh; k++) {
    const double x = __ldg(lp.gh + k), w = __ldg(lp.gh + AGP_MAX_GH_POINTS + k);
    const double f = mu + sq2sd * x;
    double ll, dll, dpar;
    loglik_d1(lp, f, y, cst, ll, dll, dpar);
    sE += w * ll;
    sM += w * dll;
    sS += w * dll * (1.4142135623730951 * x);
    sG += w * dpar;
  }
  const double isp = 0.5641895835477563;  // 1/sqrt(pi)
  double wsum = 0.0;
  if (lp.kind == AGP_LIK_GAMMA_EXP)
    for (int k = 0; k < lp.ngh; k++) wsum += __ldg(lp.gh + AGP_MAX_GH_POINTS + k);
  E = isp * sE;
  dmu = isp * sM;
  dvar = isp * sS / (2.0 * sd);
  ds2 = isp * sG + ((lp.kind == AGP_LIK_GAMMA_EXP) ? isp * wsum * (log(y) - digamma(lp.sigma2)) : 0.0);
}

}  // namespace agp
