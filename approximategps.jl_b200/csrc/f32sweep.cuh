// f32sweep.cuh -- the Float32 fast mode of the SVGP sweep (north_star "Float32 is an optional fast mode", parity 1e-4).
//
// Error budget (DESIGN.md section 8): the marginal variance k(x,x) - a^T a + c^T c cancels to ~jitter next to an inducing point, and
// an FP32-sized error in Kuf or in the forward solve is amplified by cond(Lk) into negative variances, so S1 (Kuf generator +
// A = Lk^-1 Kuf), the per-point stage, every reduction and the whole O(M^3) epilogue stay FP64.  The four GEMM-shaped stages whose
// errors enter the result additively or only through the gradient move to the tcgen05 tensor path as 3xTF32 split products
// (tf32x3.cuh) on point-major hi / lo FP32 planes:
//   S2  C[n][j]  = sum_{l >= j} A[n][l] Bt[l][j]          + per-point |c|^2                              (K-major x K-major)
//   S4  T[n][i]  = sum_{j <= i} C[n][j] Bt[i][j];  Ab = dmu (x) mt + 2 dv (T - A),  As = dv A            (K-major x K-major)
//   S6  G[i][j] += sum_n As[n][i] A[n][j]                 (MN-major x MN-major straight from the same planes, split over n)
//   S5  Kb[n][j] = sum_{i >= j} Ab[n][i] Linv[i][j] with the explicit inverse.  As a 3xTF32 product (AGP_COMPUTE_F32_TC_SOLVE) its error is
//       amplified by cond(Lk) into dZ / d theta (1.4e-4 at the C4 twin: outside the budget); the default is the same product on the INT8 tensor
//       path with exact accumulation (i8emu.cuh, 5 slices = 35 bits: EpiE5 below), measured 2.1x faster than the FP64 DMMA solve it
//       replaced (which was then removed from this mode).
#pragma once
#include "tf32x3.cuh"
#include "i8emu.cuh"

namespace agp {
namespace t5 {

// FP64 matrix [rows][ld] (inducing-major: row = inducing index, column = point) -> point-major hi / lo planes [cols][ldp]
__global__ void __launch_bounds__(256) transpose_split_kernel(const double* __restrict__ in, int64_t ld, int rows, int cols, float* __restrict__ hi,
                                                              float* __restrict__ lo, int64_t ldp) {
  __shared__ double tile[32][33];
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int j = ty; j < 32; j += 8) tile[j][tx] = (r0 + j < rows && c0 + tx < cols) ? in[(int64_t)(r0 + j) * ld + c0 + tx] : 0.0;
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j, r = r0 + tx;
    if (c < cols && r < rows) {
      float h, l;
      split_tf32(tile[tx][j], h, l);
      hi[(int64_t)c * ldp + r] = h;
      lo[(int64_t)c * ldp + r] = l;
    }
  }
}

// element-wise split of a dense FP64 array into hi / lo planes
__global__ void split_planes_kernel(const double* __restrict__ in, float* __restrict__ hi, float* __restrict__ lo, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) split_tf32(in[i], hi[i], lo[i]);
}

// g partial sums: gpart[slab][i] += sum_{n in slab} dmu[n] (Ah + Al)[n][i]; one thread per four consecutive i (float4 loads)
__global__ void __launch_bounds__(256) gvec_kernel(const float* __restrict__ Ah, const float* __restrict__ Al, int64_t ldp, int Mp, const double* __restrict__ dmu,
                                                   int ncols, int slab, double* __restrict__ gpart, int64_t slab_stride) {
  const int i4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= Mp) return;
  const int n0 = blockIdx.y * slab, n1 = min(ncols, n0 + slab);
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int n = n0; n < n1; n++) {
    const float4 h = *reinterpret_cast<const float4*>(Ah + (int64_t)n * ldp + i4);
    const float4 l = *reinterpret_cast<const float4*>(Al + (int64_t)n * ldp + i4);
    const double w = dmu[n];
    s0 = fma(w, (double)h.x + (double)l.x, s0);
    s1 = fma(w, (double)h.y + (double)l.y, s1);
    s2 = fma(w, (double)h.z + (double)l.z, s2);
    s3 = fma(w, (double)h.w + (double)l.w, s3);
  }
  double* out = gpart + (int64_t)blockIdx.y * slab_stride + i4;
  out[0] += s0;
  out[1] += s1;
  out[2] += s2;
  out[3] += s3;
}

template <class T>
__device__ __forceinline__ void store_split32(float* __restrict__ ph, float* __restrict__ pl, const T (&v)[32]) {
#pragma unroll
  for (int j = 0; j < 32; j += 4) {
    float4 h, l;
    split_tf32((double)v[j], h.x, l.x);
    split_tf32((double)v[j + 1], h.y, l.y);
    split_tf32((double)v[j + 2], h.z, l.z);
    split_tf32((double)v[j + 3], h.w, l.w);
    *reinterpret_cast<float4*>(ph + j) = h;
    *reinterpret_cast<float4*>(pl + j) = l;
  }
}

// ---- S2: C planes + partial |c|^2 per point and column tile -----------------------------------------------------------
struct EpiF2 {
  float *Ch, *Cl;
  int64_t ld;
  double* scc_part;  // [2 Mp / 128][ldp]: one partial per 64-column half
  int64_t ldp;
  struct State {
    double cc;  // FP64: the variance k(x,x) - a^T a + c^T c cancels, so the sum of squares must not add a rounding bias of its own
  };
  __device__ __forceinline__ void begin(State& st, int, int, int, int, int) const { st.cc = 0.0; }
  __device__ __forceinline__ void operator()(State& st, int tm, int tn, int, int row, int c0, const double (&v)[32]) const {
    const int64_t off = (int64_t)(tm * TM + row) * ld + tn * TN + c0;
    store_split32(Ch + off, Cl + off, v);
#pragma unroll
    for (int j = 0; j < 32; j++) st.cc = fma(v[j], v[j], st.cc);
  }
  __device__ __forceinline__ void end(State& st, int tm, int tn, int, int row, int half) const {
    scc_part[(int64_t)(2 * tn + half) * ldp + tm * TM + row] = st.cc;
  }
};

// ---- S4: acc = T = Bt C.  Ab = dmu (x) mt + 2 dv (T - A),  As = dv A ---------------------------------------------------------
// PLANES: Ab goes to hi / lo planes (the operand of the tensor-core S5); otherwise to the FP64 inducing-major matrix the FP64
// triangular solve works on (a warp's 32 points are 32 consecutive doubles of a row: coalesced).
template <bool PLANES>
struct EpiF4 {
  const float *Ah, *Al;
  float *Abh, *Abl, *Ash, *Asl;
  int64_t ld;
  const double *dmu, *dv, *mt;
  double* Ab64;
  int64_t ldk;
  double* abmax = nullptr;  // optional, per point: max_i |Ab[n][i]| (atomicMax over the column tiles; the scale of the INT8 slices of S5)
  struct State {
    double dmu, dv, mx;
  };
  __device__ __forceinline__ void begin(State& st, int tm, int, int, int row, int) const {
    const int n = tm * TM + row;
    st.dmu = dmu[n];
    st.dv = dv[n];
    st.mx = 0.0;
  }
  __device__ __forceinline__ void operator()(State& st, int tm, int tn, int, int row, int c0, const double (&v)[32]) const {
    const int i0 = tn * TN + c0;
    const int64_t off = (int64_t)(tm * TM + row) * ld + i0;
    float ab[32], as[32];
    const double dv2 = 2.0 * st.dv;
    double* p64 = Ab64 + (int64_t)i0 * ldk + tm * TM + row;
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 h = *reinterpret_cast<const float4*>(Ah + off + j);
      const float4 l = *reinterpret_cast<const float4*>(Al + off + j);
      const double a[4] = {(double)h.x + (double)l.x, (double)h.y + (double)l.y, (double)h.z + (double)l.z, (double)h.w + (double)l.w};
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const double abv = fma(st.dmu, __ldg(mt + i0 + j + q), dv2 * (v[j + q] - a[q]));
        if (PLANES) ab[j + q] = (float)abv;
        else {
          p64[(int64_t)(j + q) * ldk] = abv;
          st.mx = fmax(st.mx, fabs(abv));
        }
        as[j + q] = (float)(st.dv * a[q]);
      }
    }
    if (PLANES) store_split32(Abh + off, Abl + off, ab);
    store_split32(Ash + off, Asl + off, as);
  }
  __device__ __forceinline__ void end(State& st, int tm, int, int, int row, int) const {
    // non-negative doubles order like their bit patterns
    if (!PLANES && abmax) atomicMax(reinterpret_cast<unsigned long long*>(abmax) + tm * TM + row, (unsigned long long)__double_as_longlong(st.mx));
  }
};

// ---- S5: Kb (FP64, inducing-major [j][ldk]) for the FP64 kernel-gradient contraction ---------------------------------------------
struct EpiF5 {
  double* Kb;
  int64_t ldk;
  struct State {};
  __device__ __forceinline__ void begin(State&, int, int, int, int, int) const {}
  __device__ __forceinline__ void operator()(State&, int tm, int tn, int, int row, int c0, const double (&v)[32]) const {
    double* p = Kb + (int64_t)(tn * TN + c0) * ldk + tm * TM + row;  // a warp's 32 rows (points) are 32 consecutive doubles
#pragma unroll
    for (int j = 0; j < 32; j++) p[(int64_t)j * ldk] = v[j];
  }
  __device__ __forceinline__ void end(State&, int, int, int, int, int) const {}
};

// ---- S6: G_z (FP64 column-major, lower tiles) += tile --------------------------------------------------------------------------
struct EpiF6 {
  double* G;  // [nsplit][Mp * Mp]
  int Mp;
  struct State {};
  __device__ __forceinline__ void begin(State&, int, int, int, int, int) const {}
  __device__ __forceinline__ void operator()(State&, int tm, int tn, int z, int row, int c0, const double (&v)[32]) const {
    double* p = G + (int64_t)z * Mp * Mp + (int64_t)(tn * TN + c0) * Mp + tm * TM + row;
#pragma unroll
    for (int j = 0; j < 32; j++) p[(int64_t)j * Mp] += v[j];
  }
  __device__ __forceinline__ void end(State&, int, int, int, int, int) const {}
};

}  // namespace t5

// ---- S5 of the Float32 mode on the INT8 tensor path (i8emu.cuh, <5 slices, 64 columns>): Kb[n][j] = sum_{i >= j} Ab[n][i] Linv[i][j] ---------------
// 35-bit fixed-point operands (relative to the row maximum) with EXACT accumulation: the reverse-pass solve through the explicit inverse loses
// cond(Lk) ~ 1e3 to cancellation and another factor ~30 to the spread of magnitudes inside a row of Linv, which neither 22-bit TF32 operands
// (1.4e-4 on dZ at the C4 twin) nor four slices (28 bits: 2.7e-4) can afford inside the 1e-4 budget.
// Output: Kb (FP64, inducing-major [j][ldk]) for the FP64 kernel-gradient contraction, like EpiF5.
namespace i8e {
// ---- S1's solve of the Float32 mode: A[n][l] = sum_{l' <= l} Kuf[n][l'] Linv[l][l'] with seven slices (FP64-accurate: the marginal variance
// k(x,x) - a^T a + c^T c cancels to ~jitter, so a may not carry an FP32-sized error).  Writes A (FP64, inducing-major [l][ld]: a warp's 32 points are 32
// consecutive doubles) and, per point and per 32 inducing rows, the partial column sums a^T a and a^T mt (summed in a fixed order afterwards).
struct EpiE1 {
  double* A;
  int64_t ld;
  const double* sK;   // per point
  const double* sLi;  // per inducing row l
  const double* mt;
  double* saa_part;  // [Mp / 32][ldp]
  double* sam_part;
  int64_t ldp;
  float* Ah = nullptr;  // optional: the point-major hi / lo TF32 planes of A that S2 / S4 / S6 read (32 consecutive floats per thread), so
  float* Al = nullptr;  // that the transposing split pass over A is not needed
  int64_t ldf = 0;
  __device__ __forceinline__ void operator()(int tm, int tn, int, int row, int c0, const double (&v)[32]) const {
    const int n = tm * EM + row, l0 = tn * EN + c0;
    const double sk = sK[n] * (1.0 / 16384.0);
    double* p = A + (int64_t)l0 * ld + n;
    double a[32];
    double pa = 0.0, pm = 0.0;
#pragma unroll
    for (int j = 0; j < 32; j++) {
      a[j] = v[j] * sk * __ldg(sLi + l0 + j);
      p[(int64_t)j * ld] = a[j];
      pa = fma(a[j], a[j], pa);
      pm = fma(a[j], __ldg(mt + l0 + j), pm);
    }
    saa_part[(int64_t)(l0 >> 5) * ldp + n] = pa;
    sam_part[(int64_t)(l0 >> 5) * ldp + n] = pm;
    if (Ah) t5::store_split32(Ah + (int64_t)n * ldf + l0, Al + (int64_t)n * ldf + l0, a);
  }
};
__global__ void __launch_bounds__(256) colsum_reduce_kernel(const double* __restrict__ part, int nparts, int64_t ldp, int ncols, double* __restrict__ saa,
                                                            double* __restrict__ sam) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= ncols) return;
  double a = 0.0, m = 0.0;
  for (int p = 0; p < nparts; p++) {
    a += part[(int64_t)p * ldp + n];
    m += part[(int64_t)(nparts + p) * ldp + n];
  }
  saa[n] = a;
  sam[n] = m;
}
// ---- S2 of AGP_COMPUTE_F64_EMU: C[n][j] = sum_{l >= j} A[n][l] Bt[l][j] with seven slices (FP64-accurate).  A operand: point-major slices of A
// with one scale per point (transpose_slice_kernel), B operand: the rows of Bt^T (= columns of Bt, contiguous in the column-major copy) with one
// scale per column j.  Writes C (FP64, inducing-major [j][ld], as the DMMA kernel of S2 does) and, per point and per 32 inducing rows, the partial
// column sums c^T c that the per-point stage adds up in a fixed order.
struct EpiE2 {
  double* C;
  int64_t ld;
  const double* sA;   // per point
  const double* sBt;  // per column j
  double* scc_part;   // [Mp / 32][ldp]
  int64_t ldp;
  __device__ __forceinline__ void operator()(int tm, int tn, int, int row, int c0, const double (&v)[32]) const {
    const int n = tm * EM + row, j0 = tn * EN + c0;
    const double sa = sA[n] * (1.0 / 16384.0);
    double* p = C + (int64_t)j0 * ld + n;
    double pc = 0.0;
#pragma unroll
    for (int j = 0; j < 32; j++) {
      const double cv = v[j] * sa * __ldg(sBt + j0 + j);
      p[(int64_t)j * ld] = cv;
      pc = fma(cv, cv, pc);
    }
    scc_part[(int64_t)(j0 >> 5) * ldp + n] = pc;
  }
};
constexpr int S5_NS = 5, S5_N = 64;
struct EpiE5 {
  double* Kb;
  int64_t ldk;
  const double* sAb;  // per point
  const double* sLi;  // per column j
  __device__ __forceinline__ void operator()(int tm, int tn, int, int row, int c0, const double (&v)[32]) const {
    const int n = tm * EM + row, j0 = tn * S5_N + c0;
    const double sa = sAb[n] * (1.0 / 16384.0);
    double* p = Kb + (int64_t)j0 * ldk + n;  // a warp's 32 rows (points) are 32 consecutive doubles
#pragma unroll
    for (int j = 0; j < 32; j++) p[(int64_t)j * ldk] = v[j] * sa * __ldg(sLi + j0 + j);
  }
};
}  // namespace i8e
}  // namespace agp
