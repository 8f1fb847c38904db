// dense.cuh -- once-per-step M x M building blocks: Kuu assembly, blocked Cholesky (diagonal-block
// factorisation + inversion here, panel / trailing updates through gemm.cuh), small element-wise kernels.
// Reference counterparts: `cholesky(Symmetric(cov(fz)))` (utils.jl:17 via SVA.jl:131,181) and
// `cholesky(Symmetric(B))` (Laplace.jl:216).
#pragma once
#include "gemm.cuh"
#include "kfun.cuh"

namespace agp {

// zs = s (.) z, zn = |zs|^2 ; rows >= M are zero.  z is point-major [M][D].  zsp (optional) is the padded copy the
// Kuf generator streams: row = [zs_0 .. zs_{D-1}, 0.., zn, 0] with kuf_dp(D) + 2 doubles.
__global__ void prep_z_kernel(const double* z, double* zs, double* zn, double* zsp, int Mp, KernelParams kp) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= Mp) return;
  const int Dp = kuf_dp(kp.D), Sx = Dp + 2;
  double s = 0.0;
  for (int d = 0; d < kp.D; d++) {
    const double v = (row < kp.M) ? z[(int64_t)row * kp.D + d] * kp.s[d] : 0.0;
    zs[(int64_t)row * kp.D + d] = v;
    if (zsp) zsp[(int64_t)row * Sx + d] = v;
    s = fma(v, v, s);
  }
  zn[row] = s;
  if (zsp) {
    for (int d = kp.D; d < Sx; d++) zsp[(int64_t)row * Sx + d] = 0.0;
    zsp[(int64_t)row * Sx + Dp] = s;
  }
}

// Kuu = k(Z, Z) + jitter I on the leading M x M block, identity on the padding.  Column-major, ld = Mp.
__global__ void build_kuu_kernel(double* K, int Mp, const double* zs, const double* zn, double jitter, KernelParams kp) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;  // row
  const int b = blockIdx.y;                             // column
  if (a >= Mp) return;
  double v;
  if (a >= kp.M || b >= kp.M) {
    v = (a == b) ? 1.0 : 0.0;
  } else {
    double u;
    if (a == b && kp.kind != AGP_KERNEL_LINEAR) {
      u = 0.0;  // pairwise(d, x) has an exactly-zero diagonal
    } else if (kp.D == 1 && kp.kind != AGP_KERNEL_LINEAR) {
      const double df = zs[a] - zs[b];
      u = df * df;
    } else {
      double dot = 0.0;
      const int lo = min(a, b), hi = max(a, b);  // same operation order for (a,b) and (b,a): exactly symmetric
      for (int d = 0; d < kp.D; d++) dot = fma(zs[(int64_t)lo * kp.D + d], zs[(int64_t)hi * kp.D + d], dot);
      u = u_from_dot(kp.kind, zn[lo], zn[hi], dot);
    }
    v = kp.variance * kappa_kp(kp, u);
    if (a == b) v += jitter;
  }
  K[(int64_t)b * Mp + a] = v;
}

// K[a + b*ld] = k(x_a, y_b) for two point sets given as scaled points / squared norms (cov(f.prior, x, y));
// entries with a >= nx or b >= ny are zero.
__global__ void cross_k_kernel(double* K, int64_t ld, const double* xs, const double* xn, int nx, const double* ys, const double* yn, int ny,
                               int rows, KernelParams kp) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (a >= rows) return;
  double v = 0.0;
  if (a < nx && b < ny) {
    double u;
    if (kp.D == 1 && kp.kind != AGP_KERNEL_LINEAR) {
      const double df = xs[a] - ys[b];
      u = df * df;
    } else {
      double dot = 0.0;
      for (int d = 0; d < kp.D; d++) dot = fma(xs[(int64_t)a * kp.D + d], ys[(int64_t)b * kp.D + d], dot);
      u = u_from_dot(kp.kind, xn[a], yn[b], dot);
    }
    v = kp.variance * kappa_kp(kp, u);
  }
  K[(int64_t)b * ld + a] = v;
}

// ---- diagonal-block kernel of the blocked Cholesky -----------------------------------------------------------
// One CTA factorises a 128 x 128 diagonal block (lower triangle of src) and inverts the factor:
//   dstL  <- L (strict upper zeroed),  dstLt <- inv(L),  dstUt <- inv(L)^T        (all column-major, leading dim ld)
// info[0] = first failing global column + 1 (PosDefException).  Everything runs out of shared memory with 32-wide
// blocking so that only a dozen block-wide barriers are needed: per 32-block a warp-level factorisation of the
// diagonal, a register-resident row solve of the panel and a rank-32 trailing update; then the inverse by the
// recursive rule  inv([L11 0; L21 L22]) = [X11 0; -X22 L21 X11  X22].
constexpr int PT_LD = 129;
constexpr int PT_SMEM_BYTES = (128 * PT_LD + 64 * 65 + 128) * 8;

// Cholesky of a 32 x 32 diagonal block by one warp with the rows in registers: lane i owns row i as x[k] = A[i][j + k], a window that
// slides by one column per step, so that the pivot column is always x[0] and every register index is a compile-time constant although the
// loop over j is not unrolled.  Right-looking: after column j is scaled, x[k-1] <- x[k] - l_ij l_(j+k)j.  The scaled column reaches the other
// lanes through shared memory: every lane publishes its l_ij in two doubled buffers (one shifted by an element, so that the 31 partners
// l_(j+1)j .. l_(j+31)j start at a 16-byte aligned address whatever the parity of j) and reads them back as 16 broadcast LDS.128.  Slots that
// slide past column 31 and the entries above the diagonal carry unused values.  This warp's per-column dependency chain is the critical
// path of the whole diagonal-block kernel.  Measured on one warp alone, cycles per column: shared-memory left-looking loop 853, sliding
// window with 62 SHFL 550, with 31 LDS.64 654, with 16 LDS.128 (this form) 362; the pivot chain alone (shuffle of the pivot, rsqrt, nine
// dependent FP64 operations, 31 DFMA) is 313 (profiles/r3b_potrf32_variants.jsonl).  The other forms were removed after that measurement.
// buf: 128 doubles, 16-byte aligned.
__device__ __forceinline__ void pt_potrf32w(double* blk, int lane, double* rdiag, int col0, int* info, double* buf) {
  double x[32];
#pragma unroll
  for (int c = 0; c < 32; c++) x[c] = blk[lane * PT_LD + c];
  double* bufe = buf;       // bufe[i] = l_i (i = 0..63, wraps around)
  double* bufo = buf + 64;  // bufo[i] = l_(i+1)
  const int lo = (lane + 31) & 31;
#pragma unroll 1
  for (int j = 0; j < 32; j++) {
    const double v = x[0];
    const double d = __shfl_sync(0xffffffffu, v, j);
    if (lane == 0 && !(d > 0.0)) atomicCAS(info, 0, col0 + j + 1);
    const double y = rsqrt(d);
    const double s0 = d * y;
    const double sq = fma(fma(-s0, s0, d), 0.5 * y, s0);
    const double inv = fma(fma(-sq, y, 1.0), y, y);
    const double l0 = v * inv;
    const double lij = (lane == j) ? sq : fma(fma(-l0, sq, v), inv, l0);
    bufe[lane] = lij;
    bufe[lane + 32] = lij;
    bufo[lo] = lij;
    bufo[lo + 32] = lij;
    __syncwarp();
    const double2* b = reinterpret_cast<const double2*>(((j + 1) & 1) ? (bufo + j) : (bufe + j + 1));
#pragma unroll
    for (int k = 0; k < 15; k++) {
      const double2 p = b[k];
      x[2 * k] = fma(-lij, p.x, x[2 * k + 1]);
      x[2 * k + 1] = fma(-lij, p.y, x[2 * k + 2]);
    }
    x[30] = fma(-lij, b[15].x, x[31]);
    if (lane >= j) blk[lane * PT_LD + j] = lij;  // rows above the diagonal keep the zero they were loaded with
    if (lane == j) rdiag[j] = inv;
    __syncwarp();  // the exchange buffers are rewritten by the next step
  }
}
template <int J>
struct PtSolveRow {  // x L_d^T = a for one row held in x[] (right-looking: x[J] is final, then x[k > J] -= x[J] L[k][J])
  static __device__ __forceinline__ void run(double (&x)[32], const double* Ld, const double* rdiag) {
    x[J] *= rdiag[J];
#pragma unroll
    for (int k = J + 1; k < 32; k++) x[k] = fma(-x[J], Ld[k * PT_LD + J], x[k]);
    PtSolveRow<J + 1>::run(x, Ld, rdiag);
  }
};
template <>
struct PtSolveRow<32> {
  static __device__ __forceinline__ void run(double (&)[32], const double*, const double*) {}
};
template <int I>
struct PtInvCol {  // column `lane` of inv(L_d) in x[] (right-looking forward substitution of the unit vector e_lane)
  static __device__ __forceinline__ void run(double (&x)[32], const double* Ld, const double* rdiag, int lane) {
    x[I] = (I >= lane) ? x[I] * rdiag[I] : 0.0;
#pragma unroll
    for (int k = I + 1; k < 32; k++) x[k] = fma(-x[I], Ld[k * PT_LD + I], x[k]);
    PtInvCol<I + 1>::run(x, Ld, rdiag, lane);
  }
};
template <>
struct PtInvCol<32> {
  static __device__ __forceinline__ void run(double (&)[32], const double*, const double*, int) {}
};

// X[r0.., c0..] (sz x sz) <- -X22 * L21 * X11 with X22 = s[r0.., r0..], L21 = s[r0.., c0..], X11 = s[c0.., c0..]
// (both already inverted, upper parts zero); tb is a [sz][sz+1] scratch.  All 256 threads must call this.
__device__ __forceinline__ void pt_offdiag(double* s, double* tb, int r0, int c0, int sz) {
  constexpr int LD = PT_LD;
  const int q = sz / 4, ldt = sz + 1;
  const int t = threadIdx.x;
  const bool on = t < q * q;
  const int ti = t / q, tj = t % q;  // the thread owns elements (ti + a q, tj + b q): neighbouring lanes, neighbouring columns
  double acc[4][4];
  if (on) {
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
#pragma unroll 4
    for (int k = 0; k < sz; k++) {  // T = L21 * X11
      double av[4], bv[4];
#pragma unroll
      for (int a = 0; a < 4; a++) av[a] = s[(r0 + ti + a * q) * LD + c0 + k];
#pragma unroll
      for (int b = 0; b < 4; b++) bv[b] = s[(c0 + k) * LD + c0 + tj + b * q];
#pragma unroll
      for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
    }
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) tb[(ti + a * q) * ldt + tj + b * q] = acc[a][b];
  }
  __syncthreads();
  if (on) {
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
#pragma unroll 4
    for (int k = 0; k < sz; k++) {  // X22 * T  (X22[i][k] = 0 for k > i)
      double av[4], bv[4];
#pragma unroll
      for (int a = 0; a < 4; a++) av[a] = s[(r0 + ti + a * q) * LD + r0 + k];
#pragma unroll
      for (int b = 0; b < 4; b++) bv[b] = tb[k * ldt + tj + b * q];
#pragma unroll
      for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
    }
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) s[(r0 + ti + a * q) * LD + c0 + tj + b * q] = -acc[a][b];  // L21 was consumed before the barrier
  }
  __syncthreads();
}

#ifdef AGP_PT_TIMING
#define PT_TICK(k) if (threadIdx.x == 0) pt_ticks[k] = clock64();
__device__ long long pt_ticks[16];
#else
#define PT_TICK(k)
#endif
// nvalid: leading rows / columns of the block that hold data; the rest must be identity padding, for which the 32-blocks
// of the factorisation and of the inverse are skipped (a 20 x 20 problem costs one 32-block instead of four).
__global__ void __launch_bounds__(256) potrf_trinv128_kernel(const double* src, double* dstL, double* dstLt, double* dstUt, int64_t ld, int col0,
                                                             int* info, int nvalid) {
  extern __shared__ __align__(16) double s[];  // [128][129] + scratch [64][65]
  constexpr int N = 128, LD = PT_LD;
  double* tb = s + N * LD;
  double* rdiag = tb + 64 * 65;  // 1 / L_jj
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < N * N; i += 256) {
    const int r = i % N, c = i / N;
    s[r * LD + c] = (r >= c) ? src[(int64_t)c * ld + r] : 0.0;
  }
  __syncthreads();
  PT_TICK(0)
  // ---- Cholesky, 32-wide blocks -------------------------------------------------------------------------------
  const int nact = min(N, (nvalid + 31) & ~31);  // active leading part (multiple of 32)
  if (tid < N) rdiag[tid] = 1.0;
  __syncthreads();
  // 32-wide blocks.  16-wide blocks (a register-resident, fully unrolled 16 x 16 factorisation and a DMMA trailing update) were measured
  // and removed (profiles/r2o_pt_timing.txt): a 16 x 16 block costs 4.5 us in registers whether the rsqrt sits inside the column chain or
  // not (280 ns per column against 425 ns for the shared-memory 32-wide loop of the time), the kernel alone 88.4 -> 81.6 us, but inside the
  // factorisation -- where every launch meets a cold instruction cache and the unrolled routine is 10 KB -- C3 went from 14.05 to 14.48 ms
  // per Newton iteration.
  constexpr int PB = 32;
  for (int o = 0; o < nact; o += PB) {
    if (warp == 0) pt_potrf32w(s + o * LD + o, lane, rdiag + o, col0 + o, info, tb);  // diagonal PB x PB block
    __syncthreads();
    if (o == 0) { PT_TICK(1) }
    const int T = nact - o - PB;  // rows below the diagonal block (rows >= nact are identity padding: zero below the diagonal)
    if (tid < T) {              // panel: X L_d^T = A, one row per thread, held in registers
      double* row = s + (o + PB + tid) * LD + o;
      double x[PB];
#pragma unroll
      for (int j = 0; j < PB; j++) x[j] = row[j];
      PtSolveRow<0>::run(x, s + o * LD + o, rdiag + o);
#pragma unroll
      for (int j = 0; j < PB; j++) row[j] = x[j];
    }
    __syncthreads();
    if (o == 0) { PT_TICK(2) }
    // trailing update of the lower triangle: A[i][c] -= sum_k P[i][k] P[c][k]; a thread owns the 4 x 4 elements
    // (ti + a q, tc + b q) so that neighbouring lanes read neighbouring rows (conflict-free with ld = 129); with ti, tc < q an element with
    // b > a always lies above the diagonal, so only the 10 products with b <= a are formed
    const int q = T / 4;
    for (int mt = tid; mt < q * q; mt += 256) {
      const int ti = mt / q, tc = mt % q;
      double acc[4][4];
#pragma unroll
      for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
      const double* pi = s + (o + PB + ti) * LD + o;
      const double* pc = s + (o + PB + tc) * LD + o;
#pragma unroll 4
      for (int k = 0; k < PB; k++) {
        double av[4], bv[4];
#pragma unroll
        for (int a = 0; a < 4; a++) av[a] = pi[a * q * LD + k];
#pragma unroll
        for (int b = 0; b < 4; b++) bv[b] = pc[b * q * LD + k];
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
          for (int b = 0; b <= a; b++) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
      }
#pragma unroll
      for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b <= a; b++)
          if (tc + b * q <= ti + a * q) s[(o + PB + ti + a * q) * LD + o + PB + tc + b * q] -= acc[a][b];
    }
    __syncthreads();
    if (o == 0) { PT_TICK(3) }
  }
  PT_TICK(4)
  for (int i = tid; i < N * N; i += 256) {
    const int r = i % N, c = i / N;
    dstL[(int64_t)c * ld + r] = s[r * LD + c];
  }
  __syncthreads();
  PT_TICK(5)
  // ---- inverse: the four 32 x 32 diagonal blocks (one warp each; lane j builds column j in registers) ------------
  if (warp < 4 && warp * 32 < nact) {
    const int o = warp * 32;
    double x[32];
#pragma unroll
    for (int i = 0; i < 32; i++) x[i] = (i == lane) ? 1.0 : 0.0;
    PtInvCol<0>::run(x, s + o * LD + o, rdiag + o, lane);
    __syncwarp();  // every lane has finished reading the L rows of this block
#pragma unroll
    for (int i = 0; i < 32; i++) s[(o + i) * LD + o + lane] = x[i];
  }
  __syncthreads();
  PT_TICK(6)
  if (nact > 32) pt_offdiag(s, tb, 32, 0, 32);
  if (nact > 96) pt_offdiag(s, tb, 96, 64, 32);
  PT_TICK(7)
  if (nact > 64) pt_offdiag(s, tb, 64, 0, 64);
  PT_TICK(8)
  for (int i = tid; i < N * N; i += 256) {
    const int r = i % N, c = i / N;
    dstLt[(int64_t)c * ld + r] = s[r * LD + c];
    dstUt[(int64_t)c * ld + r] = s[c * LD + r];
  }
  PT_TICK(9)
}

// ---- small-tile GEMM for the critical chain of the blocked Cholesky -----------------------------------------------------
// Between two diagonal-block kernels the chain needs one 128 x 128 block row: L[J+1,J] = Kw[J+1,J] inv(L_JJ)^T and
// Kw[J+1,J+1] -= L[J+1,J] L[J+1,J]^T (K = 512 from a whole super-panel when J+1 opens the next one).  As two 128 x 64 tiles of the
// throughput GEMM each of these took ~20 us (two SMs busy, eight barrier-separated k-stages each); here the block is cut into sixteen
// 32 x 32 tiles (one CTA of four warps each, 2 x 2 DMMA tiles per warp, k-chunks of 32 double-buffered with cp.async).  Same operand
// conventions as gemm_kernel<A_KM, B_KN> (A(m,k) = A[m + k lda], B(k,n) = B[n + k ldb], C column-major) and the same ascending-k DMMA
// accumulation and epilogue arithmetic per element, so the result is bit-identical to it.
//   ktri:       B(k,n) = 0 for k > n (B = transpose of a lower-triangular inverse): a column tile stops at k = n0 + 32
//   lower_only: tiles strictly above the diagonal are skipped (their content is never read)
constexpr int CG_T = 32, CG_KC = 32, CG_LD = 36;  // 36 = 4 mod 16: conflict-free fragments
__global__ void __launch_bounds__(128) chain_gemm32_kernel(const double* __restrict__ A, int64_t lda, const double* __restrict__ B, int64_t ldb, int K,
                                                            int ktri, int lower_only, double* C, int64_t ldc, double alpha, double beta) {
  __shared__ __align__(16) double sm[2][2][CG_KC * CG_LD];
  const int m0 = blockIdx.x * CG_T, n0 = blockIdx.y * CG_T;
  if (lower_only && n0 > m0) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wm = (warp & 1) * 16, wn = (warp >> 1) * 16;
  const int kend = ktri ? min(K, n0 + CG_T) : K;
  const int nch = kend / CG_KC;
  auto load = [&](int buf, int k0) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int p = tid + 128 * j, k = p >> 4, c2 = (p & 15) * 2;
      cp_async16(&sm[buf][0][k * CG_LD + c2], A + (int64_t)(k0 + k) * lda + m0 + c2);
      cp_async16(&sm[buf][1][k * CG_LD + c2], B + (int64_t)(k0 + k) * ldb + n0 + c2);
    }
  };
  double acc[2][2][2];
#pragma unroll
  for (int i = 0; i < 2; i++)
#pragma unroll
    for (int j = 0; j < 2; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
  load(0, 0);
  cp_async_commit();
  for (int ch = 0; ch < nch; ch++) {
    if (ch + 1 < nch) load((ch + 1) & 1, (ch + 1) * CG_KC);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const double* sA = sm[ch & 1][0];
    const double* sB = sm[ch & 1][1];
#pragma unroll
    for (int kk = 0; kk < CG_KC; kk += 4) {
      double a[2], b[2];
#pragma unroll
      for (int mi = 0; mi < 2; mi++) a[mi] = sA[(kk + t) * CG_LD + wm + mi * 8 + g];
#pragma unroll
      for (int ni = 0; ni < 2; ni++) b[ni] = sB[(kk + t) * CG_LD + wn + ni * 8 + g];
#pragma unroll
      for (int mi = 0; mi < 2; mi++)
#pragma unroll
        for (int ni = 0; ni < 2; ni++) dmma884(acc[mi][ni], a[mi], b[ni]);
    }
    __syncthreads();  // the buffer is refilled by the load issued in the next iteration
  }
#pragma unroll
  for (int mi = 0; mi < 2; mi++)
#pragma unroll
    for (int ni = 0; ni < 2; ni++)
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int row = m0 + wm + mi * 8 + g, col = n0 + wn + ni * 8 + 2 * t + e;
        double* p = C + (int64_t)col * ldc + row;
        double v = alpha * acc[mi][ni][e];
        if (beta != 0.0) v += beta * (*p);
        *p = v;
      }
}

// out = in^T for square n x n matrices with leading dimension ld (out != in)
__global__ void transpose_kernel(const double* in, double* out, int n, int64_t ld) {
  __shared__ double tile[32][33];
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) tile[j][threadIdx.x] = in[(int64_t)(by + j) * ld + bx + threadIdx.x];
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) out[(int64_t)(bx + j) * ld + by + threadIdx.x] = tile[threadIdx.x][j];
}

__global__ void fill_kernel(double* p, int64_t n, double v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

// out[i] = sum_s in[s*stride + i]   (fixed order)
__global__ void sum_slices_kernel(const double* in, int nslices, int64_t stride, int64_t n, double* out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int k = 0; k < nslices; k++) s += in[(int64_t)k * stride + i];
    out[i] = s;
  }
}

// G (column-major, lower triangle valid) -> full symmetric
__global__ void symmetrize_from_lower_kernel(double* G, int n, int64_t ld) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
  if (r < n && r > c) G[(int64_t)r * ld + c] = G[(int64_t)c * ld + r];
}

// S <- 0.5 (S + S^T)   (two-array form: out = 0.5 (A + At) where At is the transposed copy)
__global__ void sym_average_kernel(const double* A, const double* At, double* out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = 0.5 * (A[i] + At[i]);
}

}  // namespace agp
