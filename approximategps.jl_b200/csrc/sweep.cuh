// sweep.cuh -- the data-parallel SVGP sweep kernels (per chunk of points).
//
//   S1  kuf_gen_kernel            Kuf of the launch group, written into the solution matrix (row-major)
//       + trsm_kernel<TR_RHS_FWD_SUMS>  A = Lk^-1 Kuf in place (blocked left-looking TRSM)  + column a^T a, a^T mt
//   S2  gemm + EpiS2              C  = Bt^T A       (upper-triangular operand)        + column |c|^2
//   S3  perpoint_kernel           mu, var, E[log p], dE/dmu, dE/dvar                  (HBM-bound)
//   S4  gemm + EpiS4              Ab = dmu (x) mt + 2 dv (Bt C - A),  As = dv A,  g += A dmu
//   S5  trsm_kernel<TR_RHS_BWD>   Kb = Lk^-T Ab     (in place)
//   S6  syrk_kernel               G += As A^T       (lower tiles, split over point slabs)
//   S7  kgrad_kernel              contraction of Kb with dk/dz, dk/dtheta
//
// Reference counterparts: S1 = cov(f.prior, z, x) + `_chol_lower(Kuu) \ Kuf` (SVA.jl:215-219);
// S2 = `f.data.B' * A` and diag_At_A (SVA.jl:251); S3 = marginals + expected_loglikelihood
// (SVA.jl:354-355); S4-S7 = the Zygote pullbacks of those (SURVEY.md section 7.2).
#pragma once
#include "gemm.cuh"
#include "kfun.cuh"

namespace agp {

constexpr int TR_RHS_FWD = 1, TR_RHS_BWD = 2, TR_KUF_FWD_SCALED = 3, TR_RHS_FWD_SUMS = 4;
// TR_RHS_FWD_SUMS: the forward solve of S1 on a right-hand side that kuf_gen_kernel wrote into X (in place), with S1's column
// sums a^T a and a^T mt.  The Kuf tile then costs one extra HBM write + read (0.6 GB per 151 552-point launch group, ~0.1 ms at
// the measured copy bandwidth) instead of a generator entangled with the DMMA pipeline (~0.95 ms per launch group, r01t / r2a).
// TR_KUF_FWD_SCALED (Laplace prediction, Laplace.jl:427-431): the generated rows are k(x_l, x*) scaled by rowscale[l]
// (Wsqrt) before the solve, and skd[n] = sum_l k(x_l, x*_n) dvec[l] (k' * d_loglik) is accumulated from the unscaled rows.

struct TrsmArgs {
  const double* T;  // Lt (forward) or Ut (backward): column-major Mp x Mp.  Diagonal blocks hold the
                    // inverse of the factor's diagonal block, off-diagonal blocks the negated product.
  int64_t ldt;
  int nb;     // Mp / BM
  double* X;  // [Mp][ldx] row-major: solution (and, in RHS modes, the right-hand side; in place)
  int64_t ldx;
  const double* RHS;  // RHS modes, optional: right-hand side in a separate matrix (same layout); X is then only written / re-read as solution
  // the Kuf generator (kuf_gen_kernel, TR_KUF_FWD_SCALED) and S1's column sums
  const double* pts;  // chunk's points, point-major [npts][D]
  int npts;
  const double* zsp;  // [Mp][Dp + 2] padded scaled inducing inputs with their squared norm at column Dp (prep_z_kernel)
  const double* mt;  // [Mp] whitened variational mean
  double* saa;       // [ldx] sum_m a^2 per point
  double* sam;       // [ldx] sum_m a*mt per point
  const double* rowscale;  // TR_KUF_FWD_SCALED: [Mp]
  const double* dvec;      // TR_KUF_FWD_SCALED: [Mp]
  double* skd;             // TR_KUF_FWD_SCALED: [ldx]
  KernelParams kp;
};

struct StepIter {
  int J, q, kk, cnt, nb;
  bool fwd;
  __device__ __forceinline__ void init(bool f, int nb_) {
    fwd = f;
    nb = nb_;
    J = f ? 0 : nb_ - 1;
    q = 0;
    kk = 0;
    cnt = 1 + (f ? J : nb - 1 - J);
  }
  __device__ __forceinline__ bool is_diag() const { return q == 0; }
  __device__ __forceinline__ int src() const { return q == 0 ? J : (fwd ? q - 1 : nb - q); }
  __device__ __forceinline__ bool last_in_row() const { return q == cnt - 1 && kk == BM / BK - 1; }
  __device__ __forceinline__ void next() {
    if (++kk == BM / BK) {
      kk = 0;
      if (++q == cnt) {
        q = 0;
        J += fwd ? 1 : -1;
        cnt = 1 + (fwd ? J : nb - 1 - J);
      }
    }
  }
};

// Kuf rows [row0, row0+16) x the CTA's 64 points, written as a B-operand stage tile.  The 16 x 64 scaled dot products
// z_l . x_n run on the tensor pipe: warp w owns the 8 columns 8w..8w+7 and both 8-row halves, i.e. two m8n8k4 DMMA tiles
// with ceil(D/4) k-steps each, fed straight from the padded z slab (A fragments) and x rows (B fragments); the
// ||x||^2 + ||z||^2 - 2 x.z combination, the clamp and kappa are applied to the accumulator fragment, which is stored
// as double2.  (Padded rows: kfun.cuh kuf_dp.)
__device__ __forceinline__ void gen_kuf_tile(double* __restrict__ sB, const double* __restrict__ sZ, const double* __restrict__ xs, int row0,
                                             const KernelParams& kp, int warp, int lane, const double* rowscale, const double* dvec, double (&pkd)[2]) {
  const int g = lane >> 2, t = lane & 3;
  const int D = kp.D, kind = kp.kind, Dq = kuf_dp(D), Sx = Dq + 2;
  const int c0 = warp * 8 + 2 * t;  // this thread's two columns
  const double* z0 = sZ + g * Sx;   // its two rows: g and g + 8
  const double* z1 = z0 + 8 * Sx;
  const double* xa = xs + c0 * Sx;
  const double* xb = xa + Sx;
  double u[2][2];
  if (D == 1 && kind != AGP_KERNEL_LINEAR) {
    const double d00 = xa[0] - z0[0], d01 = xb[0] - z0[0], d10 = xa[0] - z1[0], d11 = xb[0] - z1[0];
    u[0][0] = d00 * d00;
    u[0][1] = d01 * d01;
    u[1][0] = d10 * d10;
    u[1][1] = d11 * d11;
  } else {
    double acc0[2] = {0.0, 0.0}, acc1[2] = {0.0, 0.0};
    const double* xf = xs + (warp * 8 + g) * Sx + t;  // B fragment: column 8w + g, k = t
    for (int k = 0; k < Dq; k += 4) {
      const double b = xf[k];
      dmma884(acc0, z0[k + t], b);
      dmma884(acc1, z1[k + t], b);
    }
    const double xna = xa[Dq], xnb = xb[Dq], zn0 = z0[Dq], zn1 = z1[Dq];
    u[0][0] = u_from_dot(kind, xna, zn0, acc0[0]);
    u[0][1] = u_from_dot(kind, xnb, zn0, acc0[1]);
    u[1][0] = u_from_dot(kind, xna, zn1, acc1[0]);
    u[1][1] = u_from_dot(kind, xnb, zn1, acc1[1]);
  }
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int row = row0 + g + 8 * h;
    const bool valid = row < kp.M;
    double v0 = valid ? kp.variance * kappa_kp(kp, u[h][0]) : 0.0;
    double v1 = valid ? kp.variance * kappa_kp(kp, u[h][1]) : 0.0;
    const double dv = dvec[row], rsc = rowscale[row];
    pkd[0] = fma(v0, dv, pkd[0]);
    pkd[1] = fma(v1, dv, pkd[1]);
    v0 *= rsc;
    v1 *= rsc;
    *reinterpret_cast<double2*>(sB + (g + 8 * h) * BTile<B_KN>::ld + c0) = make_double2(v0, v1);
  }
}

// Blocked left-looking triangular solve on one 64-column tile per CTA.  MODE TR_KUF_FWD_SCALED generates its right-hand
// side (the scaled Kuf tile) on the fly; S = pipeline depth (4, or 3 when the z slabs of a wide input would not fit).
template <int MODE, int S>
__global__ void __launch_bounds__(NTHREADS, 2) trsm_kernel(TrsmArgs a) {
  extern __shared__ __align__(128) double smem[];
  using Cfg = StageCfg<A_KM, B_KN>;
  constexpr bool FWD = MODE == TR_KUF_FWD_SCALED;             // generator mode: the Kuf tile is built inside the pipeline
  constexpr bool SUMS = FWD || MODE == TR_RHS_FWD_SUMS;       // S1's column sums
  ThreadMap tm;
  const int tid = threadIdx.x;
  const int n0 = blockIdx.x * BN;
  const int Sx = FWD ? kuf_dp(a.kp.D) + 2 : 0;       // row length of the padded z / x rows
  const int stage_elems = Cfg::elems + BK * Sx;      // A tile | B tile | z slab
  double* xs = smem + S * stage_elems;               // [64][Sx]
  uint64_t* bar = reinterpret_cast<uint64_t*>(xs + 64 * Sx);

  if (FWD) {
    // ---- stage the X tile: TMA bulk copy into the (still unused) first pipeline stage, then scale into xs rows
    const int D = a.kp.D, Dq = kuf_dp(D);
    const int nvalid = max(0, min(BN, a.npts - n0));
    double* raw = smem;  // 64 * D doubles <= one stage
    const double* src = a.pts + (int64_t)n0 * D;
    const unsigned bytes = (unsigned)(nvalid * D * 8);
    const bool use_tma = nvalid > 0 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && ((bytes & 15) == 0);
    if (tid == 0) {
      mbar_init(bar, 1);
      fence_barrier_init();
    }
    __syncthreads();
    if (use_tma) {
      if (tid == 0) {
        mbar_expect_tx(bar, bytes);
        tma_bulk_g2s(raw, src, bytes, bar);
      }
      mbar_wait(bar, 0);
    } else {
      for (int i = tid; i < nvalid * D; i += NTHREADS) raw[i] = src[i];
      __syncthreads();
    }
    if (tid < BN) {
      double nrm = 0.0;
      for (int d = 0; d < D; d++) {
        const double v = (tid < nvalid) ? raw[tid * D + d] * a.kp.s[d] : 0.0;
        xs[tid * Sx + d] = v;
        nrm = fma(v, v, nrm);
      }
      for (int d = D; d < Sx; d++) xs[tid * Sx + d] = 0.0;
      xs[tid * Sx + Dq] = nrm;
    }
    __syncthreads();  // raw (stage 0) may be overwritten from here on
  }

  double pkd[2] = {0.0, 0.0};  // FWD: partial k' * dvec of this thread's 2 columns
  StepIter it_issue, it_cons, it_gen;
  it_issue.init(MODE != TR_RHS_BWD, a.nb);
  it_cons.init(MODE != TR_RHS_BWD, a.nb);
  it_gen.init(true, a.nb);
  const int total = (BM / BK) * a.nb * (a.nb + 1) / 2;

  ALoad<A_KM> la;
  BLoad<B_KN> lb;
  la.init(a.ldt, tid);
  lb.init(a.ldx, tid);
  auto issue = [&](int slot) {
    double* st = smem + slot * stage_elems;
    const int J = it_issue.J, L = it_issue.src(), kk = it_issue.kk;
    la.load(st, a.T + (int64_t)(L * BM + kk * BK) * a.ldt + J * BM);
    if (FWD && it_issue.is_diag()) {
      // z slab of the 16 inducing rows this stage turns into Kuf rows (contiguous in the padded copy)
      const double* zsrc = a.zsp + (int64_t)(J * BM + kk * BK) * Sx;
      for (int ch = tid; ch < BK * Sx / 2; ch += NTHREADS) cp_async16(st + Cfg::elems + ch * 2, zsrc + ch * 2);
    } else {
      const double* bsrc = (a.RHS != nullptr && it_issue.is_diag()) ? a.RHS : a.X;
      lb.load(st + Cfg::a_elems, bsrc + (int64_t)(L * BM + kk * BK) * a.ldx + n0);
    }
    it_issue.next();
  };
  auto gen = [&](int slot) {  // it_gen describes the stage living in `slot`
    double* st = smem + slot * stage_elems;
    gen_kuf_tile(st + Cfg::a_elems, st + Cfg::elems, xs, it_gen.J * BM + it_gen.kk * BK, a.kp, tm.warp, tm.lane, a.rowscale, a.dvec, pkd);
  };

  Acc acc;
  acc_zero(acc);
  // column sums a^T a and a^T mt: after every block row the 32 x 32 warp tile is folded over its rows with a halving shuffle
  // tree (7 shuffles per quantity), so that a lane carries ONE column -- ni = 2 (g >> 2 & 1) + (g >> 1 & 1), e = g & 1 -- in two
  // registers instead of the eight (ni, e) partial sums per quantity a plain per-thread accumulation would hold
  double caa = 0.0, cam = 0.0;

#pragma unroll
  for (int s = 0; s < S - 1; s++) {
    if (s < total) issue(s);
    cp_async_commit();
  }
  if (FWD) {
    // the very first stage is a generator stage: build its Kuf rows before entering the loop
    cp_async_wait<S - 2>();
    __syncthreads();
    gen(0);
    it_gen.next();
  }
  for (int step = 0; step < total; step++) {
    // FWD keeps one stage less in flight: the z slab of stage step+1 must have landed so that its Kuf rows can be
    // generated behind this stage's MMAs (the FP64 work of the generator overlaps the DMMA drain of the warp).
    if (FWD) cp_async_wait<(S >= 3 ? S - 3 : 0)>();
    else cp_async_wait<S - 2>();
    __syncthreads();
    if (step + S - 1 < total) issue((step + S - 1) % S);
    cp_async_commit();
    const double* st = smem + (step % S) * stage_elems;
    // the diagonal slot is the (triangular) inverse diagonal block: skip the k-steps in which this warp's rows are all zero
    const bool active = !it_cons.is_diag() || ((MODE == TR_RHS_BWD) ? tm.tri_active_upper(it_cons.kk * BK) : tm.tri_active_lower(it_cons.kk * BK));
    if (active) mma_stage<A_KM, B_KN>(acc, st, st + Cfg::a_elems, tm);
    if (FWD) {
      if (step + 1 < total && it_gen.is_diag()) gen((step + 1) % S);
      it_gen.next();
    }
    if (it_cons.last_in_row()) {
      const int J = it_cons.J;
      double qa[8], qm[8];  // index c = 2 ni + e
#pragma unroll
      for (int c = 0; c < 8; c++) qa[c] = qm[c] = 0.0;
#pragma unroll
      for (int mi = 0; mi < 4; mi++) {
        const int row = J * BM + tm.row(mi);
        const double mtr = SUMS ? a.mt[row] : 0.0;
        double* xr = a.X + (int64_t)row * a.ldx + n0;
#pragma unroll
        for (int ni = 0; ni < 4; ni++) {
          const double v0 = acc[mi][ni][0], v1 = acc[mi][ni][1];
          *reinterpret_cast<double2*>(xr + tm.col(ni, 0)) = make_double2(v0, v1);
          if (SUMS) {
            qa[2 * ni] = fma(v0, v0, qa[2 * ni]);
            qa[2 * ni + 1] = fma(v1, v1, qa[2 * ni + 1]);
            qm[2 * ni] = fma(v0, mtr, qm[2 * ni]);
            qm[2 * ni + 1] = fma(v1, mtr, qm[2 * ni + 1]);
          }
        }
      }
      if (SUMS) {
        const bool b2 = tm.g & 4, b1 = tm.g & 2, b0 = tm.g & 1;
#pragma unroll
        for (int j = 0; j < 4; j++) {  // fold c bit 2 over lane bit 4
          const double sa = b2 ? qa[j] : qa[j + 4], sm = b2 ? qm[j] : qm[j + 4];
          qa[j] = (b2 ? qa[j + 4] : qa[j]) + __shfl_xor_sync(0xffffffffu, sa, 16);
          qm[j] = (b2 ? qm[j + 4] : qm[j]) + __shfl_xor_sync(0xffffffffu, sm, 16);
        }
#pragma unroll
        for (int j = 0; j < 2; j++) {  // c bit 1 over lane bit 3
          const double sa = b1 ? qa[j] : qa[j + 2], sm = b1 ? qm[j] : qm[j + 2];
          qa[j] = (b1 ? qa[j + 2] : qa[j]) + __shfl_xor_sync(0xffffffffu, sa, 8);
          qm[j] = (b1 ? qm[j + 2] : qm[j]) + __shfl_xor_sync(0xffffffffu, sm, 8);
        }
        {  // c bit 0 over lane bit 2
          const double sa = b0 ? qa[0] : qa[1], sm = b0 ? qm[0] : qm[1];
          caa += (b0 ? qa[1] : qa[0]) + __shfl_xor_sync(0xffffffffu, sa, 4);
          cam += (b0 ? qm[1] : qm[0]) + __shfl_xor_sync(0xffffffffu, sm, 4);
        }
      }
      acc_zero(acc);
      __threadfence();  // the block just written is re-read through L2 (cp.async.cg) by later block rows
    }
    it_cons.next();
  }
  cp_async_wait<0>();
  if (SUMS) {
    __syncthreads();
    double* sred = smem;  // [2][4 m-warps][64]
    {
      const int col = tm.wn + (((tm.g >> 2) & 1) * 2 + ((tm.g >> 1) & 1)) * 8 + 2 * tm.t + (tm.g & 1);
      sred[(tm.wm >> 5) * 64 + col] = caa;
      sred[256 + (tm.wm >> 5) * 64 + col] = cam;
    }
    __syncthreads();
    if (tid < BN) {
      a.saa[n0 + tid] = ((sred[tid] + sred[64 + tid]) + sred[128 + tid]) + sred[192 + tid];
      a.sam[n0 + tid] = ((sred[256 + tid] + sred[320 + tid]) + sred[384 + tid]) + sred[448 + tid];
    }
    if (FWD) {
      // a thread holds the partial sums of columns 8 warp + 2 t + {0, 1} over its rows: reduce over g; no other warp
      // touches these columns
#pragma unroll
      for (int e = 0; e < 2; e++) {
        double v = pkd[e];
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (tm.g == 0) a.skd[n0 + tm.warp * 8 + 2 * tm.t + e] = v;
      }
    }
  }
}

// ---- S1, first half: Kuf = cov(f.prior, z, x) (SVA.jl:216) for one launch group, row-major [Mp][ldx] -----------------------
// One thread per point (its scaled coordinates in registers), 128 inducing rows per CTA read as shared-memory broadcasts from the
// padded scaled copy of Z (prep_z_kernel: [Dq + 2] doubles per row, squared norm at column Dq); the stores of a warp are 256
// contiguous bytes of one row.  Rows >= M are written as zeros (padding of every M x chunk operand), columns >= npts get x = 0.
struct KufGenArgs {
  double* K;
  double* DK;  // optional: variance * kappa'(u), same layout (kept for S7 so that the reverse pass neither recomputes distances nor exp)
  int64_t ldx;
  int ncols;          // columns to write (multiple of BN)
  const double* pts;  // [npts][D] raw points
  int npts;
  const double* zsp;  // [Mp][Dq + 2]
  KernelParams kp;
};
constexpr int KG_ROWS = 128, KG_COLS = 256;
template <int DMAX, int KIND>  // KIND: compile-time covariance function (AGP_KERNEL_SUM stands for sums and products: a.kp.kind tells them apart)
__global__ void __launch_bounds__(KG_COLS) kuf_gen_kernel(KufGenArgs a) {
  // z rows re-padded to DMAX + 2 doubles ([0, DMAX): coordinates, zeros beyond D; [DMAX]: squared norm) so that the distance is DMAX
  // unpredicated FMAs fed by 16-byte shared-memory broadcasts; the kernel is bound by instruction issue (r2k: 85 instructions per element
  // before this layout), not by HBM or the FP64 pipe
  constexpr int SZ = DMAX + 2;
  __shared__ __align__(16) double kgz[KG_ROWS * SZ];
  constexpr int kind = KIND;
  const int D = a.kp.D, Dq = kuf_dp(D), Sx = Dq + 2;
  const int row0 = blockIdx.y * KG_ROWS;
  const int n = blockIdx.x * KG_COLS + threadIdx.x;
  for (int i = threadIdx.x; i < KG_ROWS * SZ; i += KG_COLS) {
    const int r = i / SZ, d = i - r * SZ;
    const double* src = a.zsp + (int64_t)(row0 + r) * Sx;
    kgz[i] = d < D ? src[d] : (d == DMAX ? src[Dq] : 0.0);
  }
  double x[DMAX];
  double xn = 0.0;
#pragma unroll
  for (int d = 0; d < DMAX; d++) {
    x[d] = (d < D && n < a.npts) ? a.pts[(int64_t)n * D + d] * a.kp.s[d] : 0.0;
    xn = fma(x[d], x[d], xn);
  }
  __syncthreads();
  if (n >= a.ncols) return;
  const bool direct = D == 1 && kind != AGP_KERNEL_LINEAR;
  double* out = a.K + (int64_t)row0 * a.ldx + n;
  double* outd = a.DK ? a.DK + (int64_t)row0 * a.ldx + n : nullptr;
  const double var = a.kp.variance;
  const int rvalid = max(0, min(KG_ROWS, a.kp.M - row0));  // rows >= M are padding: zeros
  const double* z = kgz;
#pragma unroll 4
  for (int r = 0; r < rvalid; r++, z += SZ, out += a.ldx) {
    double u;
    if (direct) {
      const double df = x[0] - z[0];
      u = df * df;
    } else {
      double dot = 0.0;
#pragma unroll
      for (int d = 0; d < DMAX; d += 2) {
        const double2 zz = *reinterpret_cast<const double2*>(z + d);
        dot = fma(x[d], zz.x, dot);
        dot = fma(x[d + 1], zz.y, dot);
      }
      u = u_from_dot(kind, xn, z[DMAX], dot);
    }
    if constexpr (kind == AGP_KERNEL_SUM) {
      *out = var * kappa_kp(a.kp, u);
    } else {
      double k, dk;
      kappa_and_du_gen(kind, u, a.kp.c, k, dk);
      *out = var * k;
      if (outd) {
        *outd = var * dk;
        outd += a.ldx;
      }
    }
  }
  for (int r = rvalid; r < KG_ROWS; r++, out += a.ldx) {
    *out = 0.0;
    if (outd) {
      *outd = 0.0;
      outd += a.ldx;
    }
  }
}

// ---- S2 epilogue: store C and the per-point partial |c|^2 of this row block ---------------------------
struct EpiS2 {
  double* C;
  int64_t ldc;
  double* scc_part;  // [nb][ldp]
  int64_t ldp;
  __device__ __forceinline__ void operator()(Acc& acc, const ThreadMap& tm, int m0, int n0, double* sred) const {
    double pcc[4][2];
#pragma unroll
    for (int ni = 0; ni < 4; ni++) pcc[ni][0] = pcc[ni][1] = 0.0;
#pragma unroll
    for (int mi = 0; mi < 4; mi++) {
      double* cr = C + (int64_t)(m0 + tm.row(mi)) * ldc + n0;
#pragma unroll
      for (int ni = 0; ni < 4; ni++) {
        const double v0 = acc[mi][ni][0], v1 = acc[mi][ni][1];
        *reinterpret_cast<double2*>(cr + tm.col(ni, 0)) = make_double2(v0, v1);
        pcc[ni][0] = fma(v0, v0, pcc[ni][0]);
        pcc[ni][1] = fma(v1, v1, pcc[ni][1]);
      }
    }
#pragma unroll
    for (int ni = 0; ni < 4; ni++)
#pragma unroll
      for (int e = 0; e < 2; e++) {
        double v = pcc[ni][e];
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (tm.g == 0) sred[(tm.warp & 3) * 64 + tm.col(ni, e)] = v;
      }
    __syncthreads();
    if (threadIdx.x < BN) {
      const int t = threadIdx.x;
      scc_part[(int64_t)(m0 / BM) * ldp + n0 + t] = ((sred[t] + sred[64 + t]) + sred[128 + t]) + sred[192 + t];
    }
  }
};

// ---- S4 epilogue: acc = (Bt C) tile.  Ab = dmu (x) mt + 2 dv (acc - A);  As = dv A;  g partial ---------
struct EpiS4 {
  const double* A;
  double* Ab;
  double* As;
  int64_t ld;
  const double* dmu;
  const double* dv;
  const double* mt;
  double* gpart;  // [tiles_n][ldg]
  int64_t ldg;
  __device__ __forceinline__ void operator()(Acc& acc, const ThreadMap& tm, int m0, int n0, double* sred) const {
    double dm[4][2], dvv[4][2];
#pragma unroll
    for (int ni = 0; ni < 4; ni++) {
      const double2 a = *reinterpret_cast<const double2*>(dmu + n0 + tm.col(ni, 0));
      const double2 b = *reinterpret_cast<const double2*>(dv + n0 + tm.col(ni, 0));
      dm[ni][0] = a.x;
      dm[ni][1] = a.y;
      dvv[ni][0] = b.x;
      dvv[ni][1] = b.y;
    }
#pragma unroll
    for (int mi = 0; mi < 4; mi++) {
      const int row = m0 + tm.row(mi);
      const double mtr = mt[row];
      const int64_t off = (int64_t)row * ld + n0;
      double gp = 0.0;
#pragma unroll
      for (int ni = 0; ni < 4; ni++) {
        const int c = tm.col(ni, 0);
        const double2 a = *reinterpret_cast<const double2*>(A + off + c);
        double2 ab, as;
        ab.x = fma(dm[ni][0], mtr, 2.0 * dvv[ni][0] * (acc[mi][ni][0] - a.x));
        ab.y = fma(dm[ni][1], mtr, 2.0 * dvv[ni][1] * (acc[mi][ni][1] - a.y));
        as.x = dvv[ni][0] * a.x;
        as.y = dvv[ni][1] * a.y;
        *reinterpret_cast<double2*>(Ab + off + c) = ab;
        *reinterpret_cast<double2*>(As + off + c) = as;
        gp = fma(dm[ni][0], a.x, gp);
        gp = fma(dm[ni][1], a.y, gp);
      }
      gp += __shfl_xor_sync(0xffffffffu, gp, 1);
      gp += __shfl_xor_sync(0xffffffffu, gp, 2);
      if (tm.t == 0) sred[(tm.warp >> 2) * BM + tm.row(mi)] = gp;
    }
    __syncthreads();
    if (threadIdx.x < BM) gpart[(int64_t)(n0 / BN) * ldg + m0 + threadIdx.x] += sred[threadIdx.x] + sred[BM + threadIdx.x];
  }
};

// ---- S3: per-point stage -------------------------------------------------------------------------------
constexpr int SC_E = 0, SC_DMU = 1, SC_DKXX = 2, SC_DS2 = 3, SC_DC = 4, SC_DS = 5;  // SC_DS .. SC_DS+D-1 (the first five are written as a group)
constexpr int NSC = SC_DS + MAXD;

struct PerPointArgs {
  const double* saa;
  const double* sam;
  const double* scc_part;
  int64_t ldp;
  int nb;
  const double* pts;  // [npts][D]
  const double* y;
  int npts;  // valid points
  int ncols; // padded columns (multiple of BN) to fill with zeros beyond npts
  double scale;
  double mean_const;
  KernelParams kp;
  LikParams lp;
  double* dmu;
  double* dv;
  double* mu_out;   // optional (prediction)
  double* var_out;  // optional (prediction): variance WITHOUT the 1e-18 jitter
  double* sc_part;  // [gridDim.x][NSC] block partial sums
  int* flag;        // set to AGP_ERR_DOMAIN when a marginal variance is not positive
  int predict_only;
  long long point0;  // global index (within the evaluated batch) of this chunk's first point: Monte-Carlo counter
};

// Two consecutive points per thread (16-byte loads of the per-point operands), one fused block reduction of the five
// scalars.  grid = ceil(ncols / PP_POINTS_PER_BLOCK).
constexpr int PP_POINTS_PER_BLOCK = 512;

__device__ __forceinline__ void perpoint_one(const PerPointArgs& p, int n, bool linear, double saa, double sam, double scc, double& E, double& dmu,
                                             double& dvar, double& ds2, double& kxxfac) {
  E = dmu = dvar = ds2 = 0.0;
  kxxfac = 0.0;
  if (n >= p.npts) return;
  double kxx;
  if (linear) {
    double s = 0.0;
    for (int d = 0; d < p.kp.D; d++) {
      const double xs = p.pts[(int64_t)n * p.kp.D + d] * p.kp.s[d];
      s = fma(xs, xs, s);
    }
    kxxfac = s + p.kp.c;
    kxx = p.kp.variance * kxxfac;
  } else {
    kxxfac = p.kp.f0;  // kappa(0): 1, or sum / product of the component variances
    kxx = p.kp.variance * kxxfac;
  }
  const double mu = p.mean_const + sam;
  const double var0 = kxx - saa + scc;
  if (p.mu_out) p.mu_out[n] = mu;
  if (p.var_out) p.var_out[n] = var0;
  if (!p.predict_only) {
    const double var = var0 + 1e-18;  // AbstractGPs default jitter of f_post(x), SVA.jl:354
    if (!(var > 0.0)) atomicExch(p.flag, AGP_ERR_DOMAIN);
    expected_loglik(p.lp, mu, var, p.y[n], E, dmu, dvar, ds2, p.point0 + n);
    dmu *= p.scale;
    dvar *= p.scale;
    ds2 *= p.scale;
  }
}

__global__ void __launch_bounds__(256) perpoint_kernel(PerPointArgs p) {
  __shared__ double sred[8][5];
  __shared__ double sred1[8];
  const int n0 = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
  const bool linear = p.kp.kind == AGP_KERNEL_LINEAR;
  double E[2], dmu[2], dvar[2], ds2[2], kf[2];
  {
    double2 saa = make_double2(0.0, 0.0), sam = saa, scc = saa;
    if (n0 < p.ncols) {  // ncols is even and the operand rows are 16-byte aligned
      saa = *reinterpret_cast<const double2*>(p.saa + n0);
      sam = *reinterpret_cast<const double2*>(p.sam + n0);
      for (int j = 0; j < p.nb; j++) {
        const double2 v = *reinterpret_cast<const double2*>(p.scc_part + (int64_t)j * p.ldp + n0);
        scc.x += v.x;
        scc.y += v.y;
      }
    }
    perpoint_one(p, n0, linear, saa.x, sam.x, scc.x, E[0], dmu[0], dvar[0], ds2[0], kf[0]);
    perpoint_one(p, n0 + 1, linear, saa.y, sam.y, scc.y, E[1], dmu[1], dvar[1], ds2[1], kf[1]);
  }
  if (p.predict_only) return;
  if (n0 < p.ncols) {
    *reinterpret_cast<double2*>(p.dmu + n0) = make_double2(dmu[0], dmu[1]);
    *reinterpret_cast<double2*>(p.dv + n0) = make_double2(dvar[0], dvar[1]);
  }
  // fused, fixed-order block reduction of (E, dmu, dvar * kxxfac, ds2, dc)
  double v[5] = {E[0] + E[1], dmu[0] + dmu[1], dvar[0] * kf[0] + dvar[1] * kf[1], ds2[0] + ds2[1],
                 linear ? (dvar[0] + dvar[1]) * p.kp.variance : 0.0};
#pragma unroll
  for (int q = 0; q < 5; q++)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0)
#pragma unroll
    for (int q = 0; q < 5; q++) sred[warp][q] = v[q];
  __syncthreads();
  double* out = p.sc_part + (int64_t)blockIdx.x * NSC;
  if (threadIdx.x < 5) {
    double r = 0.0;
    for (int w = 0; w < 8; w++) r += sred[w][threadIdx.x];
    out[threadIdx.x] = r;  // SC_E, SC_DMU, SC_DKXX, SC_DS2, SC_DC are 0..4
  }
  if (linear) {
    for (int d = 0; d < p.kp.D; d++) {
      double t = 0.0;
#pragma unroll
      for (int h = 0; h < 2; h++)
        if (n0 + h < p.npts) {
          const double x = p.pts[(int64_t)(n0 + h) * p.kp.D + d];
          t += dvar[h] * 2.0 * p.kp.variance * p.kp.s[d] * x * x;
        }
      const double r = block_sum(t, sred1);
      if (threadIdx.x == 0) out[SC_DS + d] = r;
    }
  }
}

// Deterministic reduction of the per-block scalars: acc[j] += sum_b part[b][j]
__global__ void __launch_bounds__(256) scal_reduce_kernel(const double* part, int nblocks, int nsc_used, double* acc) {
  __shared__ double sred[8];
  for (int j = 0; j < nsc_used; j++) {
    double v = 0.0;
    for (int b = threadIdx.x; b < nblocks; b += blockDim.x) v += part[(int64_t)b * NSC + j];
    const double r = block_sum(v, sred);
    if (threadIdx.x == 0) acc[j] += r;
  }
}

// ---- S6: G_part[split] += As A^T on the lower-triangular tiles -------------------------------------------
struct SyrkArgs {
  const double* As;
  const double* A;
  int64_t ld;
  int ncols;   // padded point count of this chunk (multiple of BN)
  int kchunk;  // points per split (multiple of BK)
  double* G;   // [nsplit][Mp*Mp] column-major
  int Mp;
};

__global__ void __launch_bounds__(NTHREADS, 2) syrk_kernel(SyrkArgs a) {
  extern __shared__ __align__(128) double smem[];
  ThreadMap tm;
  // decode the tile index: row block ti (BM rows), column block tj (BN cols), tj <= 2*ti + 1
  int t = blockIdx.x, ti = 0;
  while (t >= 2 * ti + 2) {
    t -= 2 * ti + 2;
    ti++;
  }
  const int tj = t;
  const int split = blockIdx.y;
  const int kb = split * a.kchunk;
  const int ke = min(a.ncols, kb + a.kchunk);
  if (kb >= ke) return;
  const int m0 = ti * BM, n0 = tj * BN;
  Acc acc;
  acc_zero(acc);
  // only the lower triangle of G is used: a warp whose 32 x 32 sub-tile lies strictly above the diagonal does no MMA
  const bool needed = m0 + tm.wm + 31 >= n0 + tm.wn;
  gemm_mainloop<A_MK, B_NK>(acc, smem, a.As + (int64_t)m0 * a.ld + kb, a.ld, a.A + (int64_t)n0 * a.ld + kb, a.ld,
                            (ke - kb) / BK, tm, TRI_NONE, 0, needed);
  double* G = a.G + (int64_t)split * a.Mp * a.Mp;
#pragma unroll
  for (int mi = 0; mi < 4; mi++)
#pragma unroll
    for (int ni = 0; ni < 4; ni++)
#pragma unroll
      for (int e = 0; e < 2; e++) G[(int64_t)(n0 + tm.col(ni, e)) * a.Mp + m0 + tm.row(mi)] += acc[mi][ni][e];
}

// ---- S7: contraction of a cotangent Kb (row-major [Mp][ld], rows = inducing points, columns = points)
//          with the derivatives of k(z_l, x_n).  One warp per row, lanes stride over a slab of points.
// Per (slab, row) it accumulates  rs = sum_n W,  wx[d] = sum_n W xs_nd,  dsd[d],  dvar  with
// W = Kb * variance * kappa'(u).  kgrad_finish_kernel turns these into dZ, ds, dvariance, dc.
struct KgradArgs {
  const double* Kb;
  const double* Kf;  // FAST: the kernel values variance * kappa(u) and
  const double* DK;  //       variance * kappa'(u) that kuf_gen_kernel stored for these points (same layout as Kb)
  int64_t ld;
  const double* pts;  // [npts][D] raw points
  int npts;
  const double* zs;
  const double* zn;
  int slab;      // points per slab
  double* part;  // [nslab][Mp][stride]
  int stride;    // kgrad_stride(D) = 2*D + 3 + 2*MAXC: [rs, dvar, dc, wx[D], sum W (xs-zs)^2 [D], P[MAXC], Q[MAXC]]
  int Mp;
  KernelParams kp;
};
__host__ __device__ __forceinline__ int kgrad_stride(int D) { return 2 * D + 3 + 2 * MAXC; }
__host__ __device__ __forceinline__ int theta_size(int D) { return 2 + D + 2 * MAXC; }
constexpr int AGP_KERNEL_COMPOSITE = AGP_KERNEL_SUM;  // kgrad_kernel's KIND for both sums and products (kp.kind tells them apart)

// RW rows per warp (16 or 8 rows per CTA): the points of a slab are staged through shared memory in tiles of 256
// (scaled, with their squared norm) and shared by all rows of the CTA; each lane handles 8 points of a tile for its
// RW rows, the Kb values of a tile are fetched up front so that the HBM latency overlaps the exp / FMA work.
template <int DMAX, int RW, int KIND>
__global__ void __launch_bounds__(256, (DMAX <= 8 && RW == 1) ? 2 : 1) kgrad_kernel(KgradArgs a) {
  extern __shared__ __align__(16) double kg_smem[];  // [256][Sx]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row0 = (blockIdx.x * 8 + warp) * RW;
  const int slab = blockIdx.y;
  constexpr int kind = KIND;  // compile-time covariance function: no per-element dispatch
  const int D = a.kp.D, Dp = (D + 1) & ~1, Sx = Dp + 2;
  const bool direct = D == 1 && kind != AGP_KERNEL_LINEAR;
  const int nb = slab * a.slab, ne = min(a.npts, nb + a.slab);
  double z[RW][DMAX], znr[RW];
  bool rvalid[RW];
#pragma unroll
  for (int r = 0; r < RW; r++) {
    rvalid[r] = row0 + r < a.kp.M;
#pragma unroll
    for (int d = 0; d < DMAX; d++) z[r][d] = (d < D && rvalid[r]) ? a.zs[(int64_t)(row0 + r) * D + d] : 0.0;
    znr[r] = rvalid[r] ? a.zn[row0 + r] : 0.0;
  }
  double rs[RW], dvar[RW], dcc[RW], wx[RW][DMAX], wxx[RW][DMAX];
  constexpr bool composite = KIND == AGP_KERNEL_COMPOSITE;
  double cP[composite ? RW : 1][MAXC], cQ[composite ? RW : 1][MAXC];  // sum Kb dF/dcv[c], sum Kb dF/dca[c]
#pragma unroll
  for (int c = 0; c < MAXC; c++)
#pragma unroll
    for (int r = 0; r < (composite ? RW : 1); r++) cP[r][c] = cQ[r][c] = 0.0;
#pragma unroll
  for (int r = 0; r < RW; r++) {
    rs[r] = dvar[r] = dcc[r] = 0.0;
#pragma unroll
    for (int d = 0; d < DMAX; d++) wx[r][d] = wxx[r][d] = 0.0;
  }
  for (int t0 = nb; t0 < ne; t0 += 256) {
    __syncthreads();  // the previous tile is no longer read
    {
      const int n = t0 + threadIdx.x;
      double* xr = kg_smem + threadIdx.x * Sx;
      double nrm = 0.0;
      for (int d = 0; d < D; d++) {
        const double v = (n < ne) ? a.pts[(int64_t)n * D + d] * a.kp.s[d] : 0.0;
        xr[d] = v;
        nrm = fma(v, v, nrm);
      }
      for (int d = D; d < Sx; d++) xr[d] = 0.0;
      xr[Dp] = nrm;
    }
    __syncthreads();
    const int cnt = min(256, ne - t0);
    double kb[RW][8];
#pragma unroll
    for (int r = 0; r < RW; r++)
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int p = lane + 32 * i;
        kb[r][i] = (p < cnt && rvalid[r]) ? a.Kb[(int64_t)(row0 + r) * a.ld + t0 + p] : 0.0;
      }
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int p = lane + 32 * i;  // rows >= cnt of the tile are zero and their Kb was loaded as 0: no branch needed, so that
                                    // the eight points of a lane form one basic block and their exp / FMA chains interleave
      const double* xr = kg_smem + p * Sx;
      double xs[DMAX];
#pragma unroll
      for (int d = 0; d < DMAX; d += 2) {
        if (d < Dp) {
          const double2 v = *reinterpret_cast<const double2*>(xr + d);
          xs[d] = v.x;
          if (d + 1 < DMAX) xs[d + 1] = v.y;
        } else {
          xs[d] = 0.0;
          if (d + 1 < DMAX) xs[d + 1] = 0.0;
        }
      }
      const double xnn = xr[Dp];
#pragma unroll
      for (int r = 0; r < RW; r++) {
        double u;
        if (direct) {
          const double df = xs[0] - z[r][0];
          u = df * df;
        } else {
          double dot = 0.0;
#pragma unroll
          for (int d = 0; d < DMAX; d++) dot = fma(xs[d], z[r][d], dot);
          u = u_from_dot(kind, xnn, znr[r], dot);
        }
        double k, dk;
        const double kbv = kb[r][i];
        if constexpr (composite) {
          double pc[MAXC], qc[MAXC];
          kappa_comp(a.kp, u, k, dk, pc, qc);
#pragma unroll
          for (int c = 0; c < MAXC; c++) {
            cP[r][c] = fma(kbv, pc[c], cP[r][c]);
            cQ[r][c] = fma(kbv, qc[c], cQ[r][c]);
          }
        } else {
          kappa_and_du(kind, u, a.kp.c, k, dk);
        }
        dvar[r] = fma(kbv, k, dvar[r]);
        dcc[r] += kbv;
        const double W = kbv * a.kp.variance * dk;
        rs[r] += W;
#pragma unroll
        for (int d = 0; d < DMAX; d++) {
          const double wxd = W * xs[d];
          wx[r][d] += wxd;
          wxx[r][d] = fma(wxd, xs[d], wxx[r][d]);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < RW; r++) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], o);
      dvar[r] += __shfl_xor_sync(0xffffffffu, dvar[r], o);
      dcc[r] += __shfl_xor_sync(0xffffffffu, dcc[r], o);
#pragma unroll
      for (int d = 0; d < DMAX; d++) {
        wx[r][d] += __shfl_xor_sync(0xffffffffu, wx[r][d], o);
        wxx[r][d] += __shfl_xor_sync(0xffffffffu, wxx[r][d], o);
      }
      if constexpr (composite) {
#pragma unroll
        for (int c = 0; c < MAXC; c++) {
          cP[r][c] += __shfl_xor_sync(0xffffffffu, cP[r][c], o);
          cQ[r][c] += __shfl_xor_sync(0xffffffffu, cQ[r][c], o);
        }
      }
    }
    if (lane == 0 && rvalid[r]) {
      double* out = a.part + ((int64_t)slab * a.Mp + row0 + r) * a.stride;
      out[0] += rs[r];
      out[1] += dvar[r];
      out[2] += dcc[r];
      if constexpr (composite) {
#pragma unroll
        for (int c = 0; c < MAXC; c++) {
          out[3 + 2 * D + c] += cP[r][c];
          out[3 + 2 * D + MAXC + c] += cQ[r][c];
        }
      }
#pragma unroll
      for (int d = 0; d < DMAX; d++)
        if (d < D) {
          out[3 + d] += wx[r][d];
          // sum W (xs - zs)^2 = sum W xs^2 - 2 zs sum W xs + zs^2 sum W   (linear: sum W xs zs = zs sum W xs)
          out[3 + D + d] += (kind == AGP_KERNEL_LINEAR) ? z[r][d] * wx[r][d] : fma(z[r][d], fma(z[r][d], rs[r], -2.0 * wx[r][d]), wxx[r][d]);
        }
    }
  }
}

// S7 inside the sweep for the stationary kinds: kappa (and, for the Matern kinds, kappa') are READ BACK from what kuf_gen_kernel stored for
// these points instead of being recomputed -- no distances, no exp.  What is left per element is two or three streamed loads and 3 D + 3
// FMA-class operations, so the kernel is organised as a stream: the scaled points of half a slab are staged in shared memory once (two block
// barriers per KF_TILE points instead of two per 256), every warp then walks its row with the loads of the next 128 points in flight while it
// accumulates the current ones.  SqExponential: kappa' = -kappa / 2, only Kf is read.  Output layout = kgrad_kernel's.
template <int DMAX>
struct KfTile {
  static constexpr int value = DMAX <= 8 ? 1024 : (DMAX <= 16 ? 512 : 256);  // points staged at a time: value * (DMAX + 2) * 8 bytes <= 80 KB
};
template <int DMAX, bool SE>
__global__ void __launch_bounds__(256, DMAX <= 8 ? 2 : 1) kgrad_stream_kernel(KgradArgs a) {
  extern __shared__ __align__(16) double kf_smem[];  // [KF_TILE][Sx]
  constexpr int TILE = KfTile<DMAX>::value, U = 4;   // a lane owns U points of a 32 U-point chunk
  constexpr int Sx = DMAX + 2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + warp;
  const int slab = blockIdx.y;
  const int D = a.kp.D;
  const bool rvalid = row < a.kp.M;
  const int nb = slab * a.slab, ne = min(a.npts, nb + a.slab);
  const double* kbr = a.Kb + (int64_t)row * a.ld;
  const double* kfr = a.Kf + (int64_t)row * a.ld;
  const double* dkr = SE ? nullptr : a.DK + (int64_t)row * a.ld;
  double rs = 0.0, dvar = 0.0, wx[DMAX], wxx[DMAX];
#pragma unroll
  for (int d = 0; d < DMAX; d++) wx[d] = wxx[d] = 0.0;
  for (int t0 = nb; t0 < ne; t0 += TILE) {
    const int cnt = min(TILE, ne - t0);
    __syncthreads();  // the previous tile is no longer read
    for (int p = threadIdx.x; p < TILE; p += 256) {
      double* xr = kf_smem + p * Sx;
#pragma unroll
      for (int d = 0; d < DMAX; d++) xr[d] = (d < D && p < cnt) ? a.pts[(int64_t)(t0 + p) * D + d] * a.kp.s[d] : 0.0;
    }
    __syncthreads();
    if (!rvalid) continue;
    double kb[2][U], kf[2][U], dk[2][U];
    auto fetch = [&](int buf, int c0) {
#pragma unroll
      for (int i = 0; i < U; i++) {
        const int p = c0 + lane + 32 * i;
        const bool ok = p < cnt;
        kb[buf][i] = ok ? kbr[t0 + p] : 0.0;
        kf[buf][i] = ok ? kfr[t0 + p] : 0.0;
        if (!SE) dk[buf][i] = ok ? dkr[t0 + p] : 0.0;
      }
    };
    fetch(0, 0);
    int buf = 0;
    for (int c0 = 0; c0 < cnt; c0 += 32 * U, buf ^= 1) {
      if (c0 + 32 * U < cnt) fetch(buf ^ 1, c0 + 32 * U);
#pragma unroll
      for (int i = 0; i < U; i++) {
        const double* xr = kf_smem + (c0 + lane + 32 * i) * Sx;  // (rows >= cnt are zero and their cotangent was fetched as 0)
        const double kbv = kb[buf][i];
        dvar = fma(kbv, kf[buf][i], dvar);  // sum Kb variance kappa: divided by the variance at the end
        const double W = SE ? -0.5 * (kbv * kf[buf][i]) : kbv * dk[buf][i];
        rs += W;
#pragma unroll
        for (int d = 0; d < DMAX; d += 2) {
          const double2 v = *reinterpret_cast<const double2*>(xr + d);
          const double w0 = W * v.x, w1 = W * v.y;
          wx[d] += w0;
          wxx[d] = fma(w0, v.x, wxx[d]);
          wx[d + 1] += w1;
          wxx[d + 1] = fma(w1, v.y, wxx[d + 1]);
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    rs += __shfl_xor_sync(0xffffffffu, rs, o);
    dvar += __shfl_xor_sync(0xffffffffu, dvar, o);
#pragma unroll
    for (int d = 0; d < DMAX; d++) {
      wx[d] += __shfl_xor_sync(0xffffffffu, wx[d], o);
      wxx[d] += __shfl_xor_sync(0xffffffffu, wxx[d], o);
    }
  }
  if (lane == 0 && rvalid) {
    double* out = a.part + ((int64_t)slab * a.Mp + row) * a.stride;
    out[0] += rs;
    out[1] += dvar / a.kp.variance;
#pragma unroll
    for (int d = 0; d < DMAX; d++)
      if (d < D) {
        const double z = a.zs[(int64_t)row * D + d];
        out[3 + d] += wx[d];
        out[3 + D + d] += fma(z, fma(z, rs, -2.0 * wx[d]), wxx[d]);  // sum W (xs - zs)^2
      }
  }
}

// dZ[l][d] += zfac * (stationary: 2 s_d (zs_ld rs - wx_d) | linear: s_d wx_d);  row-wise theta partials
// are reduced over rows by thread 0 of each block into tpart, then summed by the host-side epilogue.
struct KgradFinishArgs {
  const double* part;
  int nslab;
  int Mp;
  int stride;
  const double* zs;
  double zfac;
  double* dZ;     // [Mp][D] accumulated
  double* theta;  // [theta_size(D)]: dvariance, dc, ds[d], then per component d cv[c] (MAXC) and d (component inverse lengthscale) (MAXC)
  KernelParams kp;
};

__global__ void __launch_bounds__(256) kgrad_finish_kernel(KgradFinishArgs a) {
  __shared__ double sred[8];
  const int D = a.kp.D;
  const bool linear = a.kp.kind == AGP_KERNEL_LINEAR;
  double tv = 0.0, tc = 0.0;
  // one block; threads stride over rows
  for (int j = 0; j < 2 + D; j++) {
    double v = 0.0;
    for (int row = threadIdx.x; row < a.kp.M; row += blockDim.x) {
      double s = 0.0;
      for (int sl = 0; sl < a.nslab; sl++) {
        const double* in = a.part + ((int64_t)sl * a.Mp + row) * a.stride;
        s += (j == 0) ? in[1] : (j == 1) ? in[2] : in[3 + D + (j - 2)];
      }
      v += s;
    }
    const double r = block_sum(v, sred);
    if (threadIdx.x == 0) {
      if (j == 0) tv = r;
      else if (j == 1) tc = r;
      else {
        const int d = j - 2;
        // stationary: ds_d = (2/s_d) sum W (xs-zs)^2 ; linear: (2/s_d) sum W xs zs
        a.theta[2 + d] += (a.kp.s[d] != 0.0) ? 2.0 / a.kp.s[d] * r : 0.0;
      }
    }
  }
  if (threadIdx.x == 0) {
    a.theta[0] += tv;
    a.theta[1] += linear ? a.kp.variance * tc : 0.0;
  }
  if (kernel_is_composite(a.kp.kind)) {
    // k = variance F: d/d cv[c] = variance sum Kb dF/dcv[c];  d/d s_c = variance sum Kb dF/dca[c] * 2 s_c,  ca[c] = s_c^2
    for (int j = 0; j < 2 * MAXC; j++) {
      double v = 0.0;
      for (int row = threadIdx.x; row < a.kp.M; row += blockDim.x) {
        double s = 0.0;
        for (int sl = 0; sl < a.nslab; sl++) s += a.part[((int64_t)sl * a.Mp + row) * a.stride + 3 + 2 * D + j];
        v += s;
      }
      const double r = block_sum(v, sred);
      if (threadIdx.x == 0) {
        const int c = j % MAXC;
        a.theta[2 + D + j] += (j < MAXC) ? a.kp.variance * r : a.kp.variance * r * 2.0 * sqrt(a.kp.ca[c]);
      }
    }
  }
  for (int i = threadIdx.x; i < a.kp.M * D; i += blockDim.x) {
    const int row = i / D, d = i % D;
    double rs = 0.0, wx = 0.0;
    for (int sl = 0; sl < a.nslab; sl++) {
      const double* in = a.part + ((int64_t)sl * a.Mp + row) * a.stride;
      rs += in[0];
      wx += in[3 + d];
    }
    const double sd = a.kp.s[d];
    const double g = linear ? sd * wx : 2.0 * sd * (a.zs[(int64_t)row * D + d] * rs - wx);
    a.dZ[i] += a.zfac * g;
  }
}

}  // namespace agp
