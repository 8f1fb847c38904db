// laplace.cuh -- device kernels of the Laplace Newton loop (LaplaceApproximationModule.jl:201-276, 330-369).
//
// All matrices are column-major n_p x n_p (n_p = n rounded up to 128, leading dimension n_p); the padding
// of K is zero and the padding of B = I + sqrt(W) K sqrt(W) is the identity, so padded entries of every
// vector stay exactly zero.  The O(n^3) work (cholesky(B), B^-1 for the pullback) runs on the DMMA GEMM /
// TRSM kernels of gemm.cuh / sweep.cuh; the kernels here are the O(n^2) and O(n) pieces around them.
#pragma once
#include "dense.cuh"
#include "kfun.cuh"

namespace agp {

// vector slots of the Laplace workspace (each n_p doubles)
enum { LV_F = 0, LV_FNEW, LV_Y, LV_W, LV_S, LV_DLL, LV_B, LV_CVEC, LV_U, LV_V, LV_A, LV_T0, LV_T1, LV_T2, LV_T3, LV_T4, LV_T5, LV_FBAR, LV_UBAR, LV_CBAR,
       LV_R, LV_S_NC, LV_DLL_NC, LV_X, LV_COUNT };

// ---- K8: log p(y|f), its derivatives and the Newton right-hand side -----------------------------------
// W = -d2, S = sqrt(W), b = W f + d1 (Laplace.jl:213-217); ll partial sums per block; flag on W < 0.
// d3 (third derivative) is written when requested (pullback only).
struct LapDerivArgs {
  const double* f;
  const double* y;
  int n;
  int np;
  LikParams lp;
  double* W;
  double* S;
  double* dll;
  double* b;
  double* d3;       // optional
  double* ll_part;  // [gridDim.x]
  int* flag;
};

__global__ void __launch_bounds__(256) lap_derivs_kernel(LapDerivArgs a) {
  __shared__ double sred[8];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double ll = 0.0;
  if (i < a.np) {
    double W = 0.0, d1 = 0.0, d3 = 0.0, b = 0.0;
    if (i < a.n) {
      const double f = a.f[i], y = a.y[i];
      if (a.lp.kind == AGP_LIK_BERNOULLI_LOGIT) {
        const bool one = y > 0.5;
        const double p = logistic(f);
        ll = -softplus(one ? -f : f);
        d1 = (one ? 1.0 : 0.0) - p;
        W = p * (1.0 - p);
        d3 = -p * (1.0 - p) * (1.0 - 2.0 * p);
      } else if (a.lp.kind == AGP_LIK_BERNOULLI_PROBIT) {
        // l = log Phi(z), z = s f, r = phi(z) / Phi(z): d1 = s r, d2 = -r (z + r), d3 = s r ((z + r)(z + 2 r) - 1)
        const double sg = (y > 0.5) ? 1.0 : -1.0, z = sg * f;
        double r;
        log_ndtr_and_ratio(z, ll, r);
        d1 = sg * r;
        W = r * (z + r);
        d3 = sg * r * ((z + r) * (z + 2.0 * r) - 1.0);
      } else if (a.lp.kind == AGP_LIK_POISSON_EXP) {
        const double lam = exp(f);
        ll = y * f - lam - lgamma(y + 1.0);
        d1 = y - lam;
        W = lam;
        d3 = -lam;
      } else if (a.lp.kind == AGP_LIK_EXPONENTIAL_EXP || a.lp.kind == AGP_LIK_GAMMA_EXP) {
        const double alpha = (a.lp.kind == AGP_LIK_GAMMA_EXP) ? a.lp.sigma2 : 1.0;
        const double t = y * exp(-f);  // Exponential / Gamma with scale exp(f)
        ll = loglik_const(a.lp, y) - t - alpha * f;
        d1 = -alpha + t;
        W = t;
        d3 = t;
      } else {
        const double r = y - f, s2 = a.lp.sigma2;
        ll = -0.5 * (1.8378770664093453 + log(s2)) - 0.5 * r * r / s2;
        d1 = r / s2;
        W = 1.0 / s2;
        d3 = 0.0;
      }
      if (W < 0.0) atomicExch(a.flag, AGP_ERR_DOMAIN);  // sqrt.(W) throws DomainError, Laplace.jl:214
      b = fma(W, f, d1);
    }
    a.W[i] = W;
    a.S[i] = sqrt(fmax(W, 0.0));
    a.dll[i] = d1;
    a.b[i] = b;
    if (a.d3) a.d3[i] = d3;
  }
  const double r = block_sum(ll, sred);
  if (threadIdx.x == 0) a.ll_part[blockIdx.x] = r;
}

// ---- K6: B = I + (S .* K) .* S'  (Laplace.jl:215); identity on the padding --------------------------------
__global__ void lap_build_B_kernel(const double* K, const double* S, int n, int np, double* B) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
  if (r >= np) return;
  double v = (r == c) ? 1.0 : 0.0;
  if (r < n && c < n) v += (S[r] * K[(int64_t)c * np + r]) * S[c];
  B[(int64_t)c * np + r] = v;
}

// ---- symmetric matrix-vector product: y_i = sum_j K[j + i*ld] x_j (one warp per column) ------------------
// Optional element-wise companions: K2 != NULL multiplies entry-wise (y_i = sum_j K_ji K2_ji x_j).
__global__ void __launch_bounds__(256) symv_kernel(const double* K, const double* K2, int64_t ld, int n, const double* x, double* y) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + warp;
  if (i >= n) return;
  const double* col = K + (int64_t)i * ld;
  const double* col2 = K2 ? K2 + (int64_t)i * ld : nullptr;
  double acc0 = 0.0, acc1 = 0.0;
  int j = lane;
  for (; j + 32 < n; j += 64) {
    acc0 = fma(col2 ? col[j] * col2[j] : col[j], x[j], acc0);
    acc1 = fma(col2 ? col[j + 32] * col2[j + 32] : col[j + 32], x[j + 32], acc1);
  }
  if (j < n) acc0 = fma(col2 ? col[j] * col2[j] : col[j], x[j], acc0);
  double acc = acc0 + acc1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) y[i] = acc;
}

// ---- blocked triangular solves with a vector right-hand side (one launch per 128-block) ------------------
// Forward, L x = b:  x_J = inv(L_JJ) b_J, then b_I -= L_IJ x_J for the block rows I > J (one CTA each).
// Linv holds inv(L_JJ) in its diagonal blocks (column-major).  CTA 0 only publishes x_J.
__global__ void __launch_bounds__(256) trsv_fwd_step_kernel(const double* L, const double* Linv, int64_t ld, int J, double* b, double* x) {
  __shared__ double xj[128];
  __shared__ double part[256];
  const int tid = threadIdx.x, i = tid & 127, h = tid >> 7;
  {
    const double* inv = Linv + (int64_t)J * 128 * ld + (int64_t)J * 128;
    const double* bj = b + (int64_t)J * 128;
    double acc = 0.0;
    for (int k = h * 64; k < h * 64 + 64; k++) acc = fma(inv[i + (int64_t)k * ld], bj[k], acc);
    part[tid] = acc;
    __syncthreads();
    if (tid < 128) xj[tid] = part[tid] + part[tid + 128];
    __syncthreads();
  }
  if (blockIdx.x == 0) {
    if (tid < 128) x[(int64_t)J * 128 + tid] = xj[tid];
    return;
  }
  const int64_t r = (int64_t)(J + blockIdx.x) * 128 + i;
  const double* Lp = L + (int64_t)J * 128 * ld + r;
  double acc = 0.0;
  for (int k = h * 64; k < h * 64 + 64; k++) acc = fma(Lp[(int64_t)k * ld], xj[k], acc);
  part[tid] = acc;
  __syncthreads();
  if (tid < 128) b[r] -= part[tid] + part[tid + 128];
}

// Backward, L^T x = b:  x_J = inv(L_JJ)^T b_J, then b_c -= sum_i L[J*128+i, c] x_J[i] for the columns c of
// the block columns < J (one CTA per block column, one warp per 16 columns).  LinvT holds inv(L_JJ)^T.
__global__ void __launch_bounds__(256) trsv_bwd_step_kernel(const double* L, const double* LinvT, int64_t ld, int J, double* b, double* x) {
  __shared__ double xj[128];
  __shared__ double part[256];
  const int tid = threadIdx.x, i = tid & 127, h = tid >> 7;
  {
    const double* inv = LinvT + (int64_t)J * 128 * ld + (int64_t)J * 128;
    const double* bj = b + (int64_t)J * 128;
    double acc = 0.0;
    for (int k = h * 64; k < h * 64 + 64; k++) acc = fma(inv[i + (int64_t)k * ld], bj[k], acc);
    part[tid] = acc;
    __syncthreads();
    if (tid < 128) xj[tid] = part[tid] + part[tid + 128];
    __syncthreads();
  }
  if (blockIdx.x == 0) {
    if (tid < 128) x[(int64_t)J * 128 + tid] = xj[tid];
    return;
  }
  const int warp = tid >> 5, lane = tid & 31;
  const int c0 = (blockIdx.x - 1) * 128 + warp * 16;
  const double x0 = xj[lane], x1 = xj[lane + 32], x2 = xj[lane + 64], x3 = xj[lane + 96];
  for (int cc = 0; cc < 16; cc++) {
    const int c = c0 + cc;
    const double* Lp = L + (int64_t)c * ld + (int64_t)J * 128;
    double acc = fma(Lp[lane], x0, fma(Lp[lane + 32], x1, fma(Lp[lane + 64], x2, Lp[lane + 96] * x3)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) b[c] -= acc;
  }
}

// ---- single-launch blocked triangular solves (one CTA per 128-block, flag-chained) ------------------------------
// CTA J accumulates  b_J - sum_{L before J} (block J,L) x_L  as the x_L are published, applies the inverse diagonal
// block and publishes x_J.  A CTA only ever waits for CTAs with a smaller block index, which the hardware schedules
// first -- made independent of the hardware's dispatch order by a ticket: a CTA takes its block index from an atomic counter when it
// starts, so every block with a smaller index belongs to a CTA that is already running or done, whatever the occupancy and whichever
// order the block scheduler uses; the CTA that draws the last ticket resets the counter for the next launch.  `epoch` distinguishes
// successive solves without clearing the flags.
__device__ __forceinline__ int trsv_ticket(int* ticket) {
  __shared__ int s_ticket;
  if (threadIdx.x == 0) {
    const int t = atomicAdd(ticket, 1);
    if (t == (int)gridDim.x - 1) atomicExch(ticket, 0);
    s_ticket = t;
  }
  __syncthreads();
  return s_ticket;
}
__device__ __forceinline__ void trsv_wait(volatile int* flag, int epoch) {
  if (threadIdx.x == 0) {
    while (*flag != epoch) {
    }
    __threadfence();
  }
  __syncthreads();
}
__device__ __forceinline__ void trsv_publish(int* flag, int epoch) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) atomicExch(flag, epoch);
}

// L x = b.  Linv: inverse diagonal blocks (column-major).  grid = nb, block = 256.
__global__ void __launch_bounds__(256) trsv_fwd_chain_kernel(const double* L, const double* Linv, int64_t ld, const double* b, double* x, int* flags,
                                                             int epoch, int* ticket) {
  __shared__ double xs[128];
  __shared__ double part[256];
  const int J = trsv_ticket(ticket), tid = threadIdx.x, i = tid & 127, h = tid >> 7;
  double acc = 0.0;
  for (int Lb = 0; Lb < J; Lb++) {
    // the block of L does not depend on x: fetch it before waiting
    const double* Lp = L + (int64_t)(Lb * 128 + h * 64) * ld + (int64_t)J * 128 + i;
    double lv[64];
#pragma unroll
    for (int k = 0; k < 64; k++) lv[k] = __ldg(Lp + (int64_t)k * ld);
    trsv_wait(flags + Lb, epoch);
    if (tid < 128) xs[tid] = __ldcg(x + (int64_t)Lb * 128 + tid);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 64; k++) acc = fma(lv[k], xs[h * 64 + k], acc);
    __syncthreads();  // xs is rewritten in the next round
  }
  part[tid] = acc;
  __syncthreads();
  if (tid < 128) xs[tid] = b[(int64_t)J * 128 + tid] - (part[tid] + part[tid + 128]);
  __syncthreads();
  const double* inv = Linv + (int64_t)J * 128 * ld + (int64_t)J * 128;
  double a2 = 0.0;
  for (int k = h * 64; k < h * 64 + 64; k++) a2 = fma(inv[i + (int64_t)k * ld], xs[k], a2);
  part[tid] = a2;
  __syncthreads();
  if (tid < 128) x[(int64_t)J * 128 + tid] = part[tid] + part[tid + 128];
  trsv_publish(flags + J, epoch);
}

// L^T x = b.  LinvT: inverse-transposed diagonal blocks.  Block J = nb-1-blockIdx.x waits for the blocks after it.
__global__ void __launch_bounds__(256) trsv_bwd_chain_kernel(const double* L, const double* LinvT, int64_t ld, int nb, const double* b, double* x, int* flags,
                                                             int epoch, int* ticket) {
  __shared__ double xs[128];
  __shared__ double part[256];
  __shared__ double colacc[128];
  const int J = nb - 1 - trsv_ticket(ticket), tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, i = tid & 127, h = tid >> 7;
  if (tid < 128) colacc[tid] = 0.0;
  for (int Lb = nb - 1; Lb > J; Lb--) {
    // (block Lb,J)^T x_Lb: column c of the block is contiguous over the rows; one warp handles 16 columns.  The block does
    // not depend on x: fetch it into registers before waiting (the wait for x_{J+1} is the critical path of the chain)
    double lv[16][4];
#pragma unroll
    for (int cc = 0; cc < 16; cc++) {
      const double* Lp = L + (int64_t)(J * 128 + warp * 16 + cc) * ld + (int64_t)Lb * 128 + lane;
#pragma unroll
      for (int k = 0; k < 4; k++) lv[cc][k] = __ldg(Lp + 32 * k);
    }
    trsv_wait(flags + Lb, epoch);
    if (tid < 128) xs[tid] = __ldcg(x + (int64_t)Lb * 128 + tid);
    __syncthreads();
    const double x0 = xs[lane], x1 = xs[lane + 32], x2 = xs[lane + 64], x3 = xs[lane + 96];
#pragma unroll
    for (int cc = 0; cc < 16; cc++) {
      double acc = fma(lv[cc][0], x0, fma(lv[cc][1], x1, fma(lv[cc][2], x2, lv[cc][3] * x3)));
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) colacc[warp * 16 + cc] += acc;
    }
    __syncthreads();
  }
  __syncthreads();
  if (tid < 128) xs[tid] = b[(int64_t)J * 128 + tid] - colacc[tid];
  __syncthreads();
  const double* inv = LinvT + (int64_t)J * 128 * ld + (int64_t)J * 128;
  double a2 = 0.0;
  for (int k = h * 64; k < h * 64 + 64; k++) a2 = fma(inv[i + (int64_t)k * ld], xs[k], a2);
  part[tid] = a2;
  __syncthreads();
  if (tid < 128) x[(int64_t)J * 128 + tid] = part[tid] + part[tid + 128];
  trsv_publish(flags + J, epoch);
}

// ---- small vector kernels ------------------------------------------------------------------------------
// op 0: out = a .* b      op 1: out = a - b .* c      op 2: out = a ./ b (0 where b == 0 and a == 0)
__global__ void lap_vec_kernel(int op, const double* a, const double* b, const double* c, double* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double v;
  if (op == 0) v = a[i] * b[i];
  else if (op == 1) v = a[i] - b[i] * c[i];
  else v = (b[i] == 0.0 && a[i] == 0.0) ? 0.0 : a[i] / b[i];
  out[i] = v;
}

// out[0] = |f - fnew|^2, out[1] = |f|^2, out[2] = |fnew|^2  (isapprox(f, fnew), Laplace.jl:267); one block
__global__ void __launch_bounds__(256) lap_conv_kernel(const double* f, const double* fnew, int n, double* out) {
  __shared__ double sred[8];
  double d = 0.0, a = 0.0, b = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double x = f[i], y = fnew[i], e = x - y;
    d = fma(e, e, d);
    a = fma(x, x, a);
    b = fma(y, y, b);
  }
  const double rd = block_sum(d, sred), ra = block_sum(a, sred), rb = block_sum(b, sred);
  if (threadIdx.x == 0) {
    out[0] = rd;
    out[1] = ra;
    out[2] = rb;
  }
}

// out[0] = -a'f/2 + sum(ll_part) - sum(log diag L)   (_laplace_lml, Laplace.jl:250-254); one block
__global__ void __launch_bounds__(256) lap_lml_kernel(const double* a, const double* f, const double* L, int64_t ld, int n, const double* ll_part,
                                                      int nparts, double* out) {
  __shared__ double sred[8];
  double af = 0.0, ld_ = 0.0, ll = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    af = fma(a[i], f[i], af);
    ld_ += log(L[(int64_t)i * ld + i]);
  }
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) ll += ll_part[i];
  const double r0 = block_sum(af, sred), r1 = block_sum(ld_, sred), r2 = block_sum(ll, sred);
  if (threadIdx.x == 0) {
    out[0] = -0.5 * r0 + r2 - r1;
    out[1] = r2;
  }
}

// ---- pullback vector stages (oracle/laplace.py lml_and_grad_K, op by op) ----------------------------------
// stage 0 (before the solves):  vbar = S f / 2 -> T0
// stage 1 (after ubar = B^-1 vbar):  cbar = S ubar;  T1 = v S;  T2 = ubar S
// stage 2 (after t1 = (Binv.*K) S -> T0, t2 = K (v S) -> T4, t3 = K (ubar S) -> T5, kc = K cbar -> T3; d3 in X):
//          sbar = f v / 2 + ubar cvec - t1 - ubar t2 - v t3
//          bbar = -f/2 + kc
//          Wbar = bbar f + sbar / (2 S);  fbar = -a/2 + dll + W bbar + bbar (-W) - Wbar d3   -> FBAR;  R0 = fbar ./ S_nc
struct LapBackArgs {
  double* v[LV_COUNT];
  int n;
};
__global__ void lap_back_kernel(int stage, LapBackArgs p) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  double** v = p.v;
  if (stage == 0) {
    v[LV_T0][i] = 0.5 * v[LV_S][i] * v[LV_F][i];
  } else if (stage == 1) {
    const double s = v[LV_S][i], ub = v[LV_UBAR][i];
    v[LV_CBAR][i] = s * ub;
    v[LV_T1][i] = v[LV_V][i] * s;
    v[LV_T2][i] = ub * s;
  } else {
    const double s = v[LV_S][i], f = v[LV_F][i], vv = v[LV_V][i], ub = v[LV_UBAR][i], W = v[LV_W][i];
    const double sbar = 0.5 * f * vv + ub * v[LV_CVEC][i] - v[LV_T0][i] - ub * v[LV_T4][i] - vv * v[LV_T5][i];
    const double bbar = -0.5 * f + v[LV_T3][i];
    const double Wbar = bbar * f + ((s == 0.0 && sbar == 0.0) ? 0.0 : sbar / (2.0 * s));
    // fbar = (-a/2 + g) + W bbar + gbar h + hbar d3   with gbar = bbar, h = -W, hbar = -Wbar
    const double fbar = -0.5 * v[LV_A][i] + v[LV_DLL][i] + W * bbar + bbar * (-W) - Wbar * v[LV_X][i];
    v[LV_FBAR][i] = fbar;
    const double snc = v[LV_S_NC][i];
    v[LV_R][i] = (snc == 0.0 && fbar == 0.0) ? 0.0 : fbar / snc;
  }
}

// Kbar[i,j] = cbar_i b_j - S_i Binv_ij S_j / 2 - S_i ubar_i v_j S_j + r_i g_j   (column-major, ld = np)
// sym != 0 writes the symmetrised (Kbar + Kbar^T)/2 instead (what the kernel-parameter contraction needs).
__global__ void lap_kbar_kernel(const double* Binv, int64_t ld, int n, int np, const double* cbar, const double* b, const double* S, const double* ubar,
                                const double* v, const double* r, const double* g, int sym, double* Kbar) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= np) return;
  double out = 0.0;
  if (i < n && j < n) {
    const double core = -0.5 * S[i] * Binv[(int64_t)j * ld + i] * S[j];
    const double a_ij = fma(cbar[i], b[j], fma(-(S[i] * ubar[i]), v[j] * S[j], r[i] * g[j]));
    if (sym) {
      const double a_ji = fma(cbar[j], b[i], fma(-(S[j] * ubar[j]), v[i] * S[i], r[j] * g[i]));
      out = core + 0.5 * (a_ij + a_ji);
    } else {
      out = core + a_ij;
    }
  }
  Kbar[(int64_t)j * ld + i] = out;
}

}  // namespace agp
