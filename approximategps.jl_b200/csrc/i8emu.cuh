// i8emu.cuh -- FP64-accurate products on the INT8 tensor path (Ozaki-style error-free slicing), experimental engine.
//
//   C[m][n] = sum_k A[m][k] B[n][k]      A, B given as S = 7 signed 7-bit slices per element plus one power-of-two scale per row:
//       x = 2^e(row) * sum_{i<S} q_i 2^{-7(i+1)},   q_i in [-127, 127]   (slice7(): exact in FP64; the residual, < 2^-49 of the row maximum, is dropped)
//   so that every slice product q_i^A q_j^B is an exact integer and the 28 products with i + j <= S - 1 are accumulated EXACTLY by
//   tcgen05.mma.kind::i8 into INT32 accumulators in TMEM -- one accumulator per g = i + j (all products of a group share the scale
//   2^{-7(g+2)}), 7 x 64 = 448 of the 512 TMEM columns of a CTA.  The groups are recombined in FP64 by the epilogue.  What is lost
//   against an FP64 FMA chain: the dropped residuals and the dropped products with i + j >= S, both below 2^-46 of (row max of A) x
//   (row max of B) per term -- a normwise bound, like a blocked DGEMM's, with a constant 4e3 times smaller than cond * eps of the solves
//   around it.  FP64 DMMA and DFMA share one 37 TFLOP/s ceiling on B200; the INT8 path is 4.5 POPS, i.e. 160 TFLOP/s FP64-equivalent at
//   28 products.
//
// One CTA computes one 128 x 64 output tile over its k-range:
//   warp 0      TMA producer: per k-block of 128 the 7 B-slice tiles (64 x 128 B each, one mbarrier, double-buffered) and then the 7 A-slice
//               tiles (128 x 128 B) one by one through a 4-slot ring; 128-byte swizzle, K-major, 3-D tensor maps (k, row, slice)
//   warp 1      one elected thread issues, per A-slice i, the products with B-slices j <= S-1-i into accumulator i + j (4 MMAs of k = 32 each)
//               and commits the ring slot back; after the last k-block it commits the accumulators to the epilogue
//   warps 2..5  epilogue: tcgen05.ld of the 7 accumulators of this thread's row, FP64 recombination sum_g acc_g 2^{-7g}, functor
// SASS: UTCIMMA, LDTM, UTMALDG.
#pragma once
#include "tf32x3.cuh"

namespace agp {
namespace i8e {

using t5::mbar_expect_tx_u32;
using t5::mbar_init_u32;
using t5::mbar_wait_u32;
using t5::smem_u32;
using t5::tc_commit;
using t5::tc_fence_after;
using t5::tc_fence_before;

constexpr int S = 7;     // slices per operand of the FP64-accurate configuration (49 bits)
constexpr int EM = 128;  // output rows per CTA = TMEM lanes
constexpr int EN = 64;   // output columns per CTA (per accumulator group) of the S = 7 configuration: 7 x 64 = 448 TMEM columns
constexpr int EK = 128;  // k per pipeline stage = one 128-byte swizzle row of int8
constexpr int UK = 32;   // k of one tcgen05.mma.kind::i8
constexpr int A_TILE = EM * EK;
constexpr int A_SLOTS = 4;
constexpr int E_THREADS = 64 + 128;
constexpr int TMEM_COLS = 512;
// Configuration <NS slices, N columns>: NS * N <= 512 TMEM columns.  <7, 64>: FP64-accurate (2^-49); <4, 128>: 28 bits -- enough for the
// Float32 mode's reverse-pass solve, whose 1e-4 budget 22-bit TF32 operands miss by the condition number -- at the full 64-cycle MMA rate.
template <int NS, int N>
struct Cfg {
  static_assert(NS * N <= TMEM_COLS && N % 32 == 0, "accumulators must fit tensor memory");
  static constexpr int b_tile = N * EK;
  static constexpr int b_stage = NS * b_tile;
  static constexpr int smem_bytes = A_SLOTS * A_TILE + 2 * b_stage + 1024 /* alignment slack */ + 256 /* barriers */;
  static constexpr int products = NS * (NS + 1) / 2;
};
constexpr int B_TILE = Cfg<S, EN>::b_tile, B_STAGE = Cfg<S, EN>::b_stage, SMEM_BYTES = Cfg<S, EN>::smem_bytes;

constexpr int KM_FULL = 0, KM_FROM_N = 1, KM_UPTO_N = 2, KM_SPLIT = 3;

struct Args {
  int K;       // contraction length (multiple of 128 in the stored planes)
  int kmode;   // KM_FROM_N: k >= tile_n * EN (B lower triangular stored [n][k]);  KM_UPTO_N: k < (tile_n + 1) * EN;  KM_SPLIT: blockIdx.z slabs
  int kchunk;  // KM_SPLIT: k per slab (multiple of 128; <= 16384 keeps 7 * 127^2 * k below 2^31)
  int lower_only;
};

// x = scale * sum_i q_i 2^{-7(i+1)}: inv_scale = 2^-e with |x| 2^-e < 1.  Every operation is exact in FP64.
template <int NS>
__host__ __device__ __forceinline__ void slice_n(double x, double inv_scale, signed char (&q)[NS]) {
  double t = x * inv_scale;
#pragma unroll
  for (int i = 0; i < NS; i++) {
    t *= 128.0;
    const double qi = trunc(t);
    q[i] = (signed char)(int)qi;
    t -= qi;
  }
}
// Round-to-nearest (signed-digit) slicing: q_i = rint(t), residual in [-1/2, 1/2], so every digit after the first is a zero-mean quantity in
// [-64, 64] and both the dropped residual and the dropped slice products (i + j >= NS) are unbiased -- over the 1.5e5 points of a launch group a
// truncation bias adds up linearly, a rounding error like sqrt(n).  Needs |x| * inv_scale <= 1/2 (first digit <= 64), i.e. twice pow2_scale().
template <int NS>
__host__ __device__ __forceinline__ void slice_rn(double x, double inv_scale, signed char (&q)[NS]) {
  double t = x * inv_scale;
#pragma unroll
  for (int i = 0; i < NS; i++) {
    t *= 128.0;
    const double qi = rint(t);
    q[i] = (signed char)(int)qi;
    t -= qi;
  }
}
__host__ __device__ __forceinline__ void slice7(double x, double inv_scale, signed char (&q)[S]) { slice_n<S>(x, inv_scale, q); }
// power-of-two scale of a row whose largest magnitude is mx: 2^e with mx 2^-e in [0.5, 1)
__host__ __device__ __forceinline__ double pow2_scale(double mx) {
  if (!(mx > 0.0)) return 1.0;
  int e;
  frexp(mx, &e);
  return ldexp(1.0, e);
}

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n" ::"r"(dst), "l"(map),
               "r"(bar), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// `leader` predicates the instruction itself: the issuing warp runs its loops convergently (warp-uniform control flow, descriptors in uniform
// registers) and one elected lane issues -- a divergent `if (lane == 0)` around the loop makes the compiler wrap every uniform-datapath
// instruction in an ELECT / BRA.U.ANY retry loop (13 instructions and ~95 cycles per MMA in the first version of this kernel)
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate, uint32_t leader) {
  asm volatile(
      "{\n"
      ".reg .pred p, q;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "setp.ne.b32 q, %5, 0;\n"
      "@q tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
using t5::elect_one;
using t5::tc_commit_pred;
__device__ __forceinline__ void tc_ld32_i(uint32_t taddr, int (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, "
      "%22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]),
        "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
        "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}
// K-major tile [rows][128 B], 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart (same descriptor as the TF32 engine's K-major one)
__device__ __forceinline__ uint64_t kdesc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor: D = S32, A = B = signed 8 bit, K-major both, M = 128, N columns, dense
__host__ __device__ constexpr uint32_t idesc_i8(int n = EN) { return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(EM >> 4) << 24); }

// Epi: operator()(tile_m, tile_n, z, row, c0, const double (&v)[32]) -- a thread owns output row `row` (0..127 of the tile) and is called
// for c0 = 0 and 32; v = sum_g acc_g 2^{-7g} (exact integers scaled by powers of two, summed in FP64); the functor applies
// 2^-14 * scaleA[row] * scaleB[col] and whatever the stage needs.
template <class Epi, int NS = S, int EN = i8e::EN>
__global__ void __launch_bounds__(E_THREADS, 1) i8emu_gemm_kernel(const __grid_constant__ CUtensorMap mA, const __grid_constant__ CUtensorMap mB, Args g, Epi epi) {
  constexpr int S = NS, B_TILE = Cfg<NS, EN>::b_tile, B_STAGE = Cfg<NS, EN>::b_stage;  // (shadow the FP64 configuration's constants)
  extern __shared__ uint8_t e_smem_raw[];
  // n-tile = fast grid index: the N / 64 CTAs that share an A row-tile (7 x 128 x K bytes) run together and read it from HBM once, through L2
  // (with the m-tile as the fast index every n-tile streamed all of A again: 16 x 1.1 GB per launch at the sweep's shape, i.e. DRAM-bound)
  const int tile_n = blockIdx.x, tile_m = blockIdx.y, z = blockIdx.z;
  if (g.lower_only && tile_n * EN >= (tile_m + 1) * EM) return;
  int kb0 = 0, ke = g.K;
  if (g.kmode == KM_FROM_N) kb0 = (tile_n * EN) & ~(EK - 1);
  if (g.kmode == KM_UPTO_N) ke = min(g.K, ((tile_n + 1) * EN + EK - 1) & ~(EK - 1));
  if (g.kmode == KM_SPLIT) {
    kb0 = z * g.kchunk;
    ke = min(g.K, kb0 + g.kchunk);
  }
  const int nk = max(0, (ke - kb0 + EK - 1) / EK);

  const uint32_t base = (smem_u32(e_smem_raw) + 1023u) & ~1023u;
  const uint32_t a_ring = base, b_stage = base + A_SLOTS * A_TILE;
  const uint32_t bars = b_stage + 2 * B_STAGE;
  auto afull = [&](int s) { return bars + 8u * s; };
  auto aempty = [&](int s) { return bars + 8u * (A_SLOTS + s); };
  auto bfull = [&](int b) { return bars + 8u * (2 * A_SLOTS + b); };
  auto bempty = [&](int b) { return bars + 8u * (2 * A_SLOTS + 2 + b); };
  const uint32_t tfull = bars + 8u * (2 * A_SLOTS + 4);
  const uint32_t tmem_slot = bars + 8u * (2 * A_SLOTS + 5);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(e_smem_raw + (tmem_slot - smem_u32(e_smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < A_SLOTS; s++) {
      mbar_init_u32(afull(s), 1);
      mbar_init_u32(aempty(s), 1);
    }
    for (int b = 0; b < 2; b++) {
      mbar_init_u32(bfull(b), 1);
      mbar_init_u32(bempty(b), 1);
    }
    mbar_init_u32(tfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(tmem_slot), "r"((uint32_t)TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_slot_ptr;

  if (warp == 0) {
    if (lane == 0 && nk > 0) {
      int ause = 0;
      for (int kb = 0; kb < nk; kb++) {
        const int buf = kb & 1, k0 = kb0 + kb * EK;
        if (kb >= 2) mbar_wait_u32(bempty(buf), ((kb >> 1) - 1) & 1);
        mbar_expect_tx_u32(bfull(buf), B_STAGE);
#pragma unroll
        for (int j = 0; j < S; j++) tma_load_3d(b_stage + buf * B_STAGE + j * B_TILE, &mB, bfull(buf), k0, tile_n * EN, j);
        for (int i = 0; i < S; i++, ause++) {
          const int slot = ause % A_SLOTS;
          if (ause >= A_SLOTS) mbar_wait_u32(aempty(slot), ((ause / A_SLOTS) - 1) & 1);
          mbar_expect_tx_u32(afull(slot), A_TILE);
          tma_load_3d(a_ring + slot * A_TILE, &mA, afull(slot), k0, tile_m * EM, i);
        }
      }
    }
  } else if (warp == 1) {
    if (nk > 0) {  // the whole warp walks the loops (uniform control flow); one elected lane issues
      const uint32_t leader = elect_one();
      constexpr uint32_t idesc = idesc_i8(EN);
      int ause = 0;
      for (int kb = 0; kb < nk; kb++) {
        const int buf = kb & 1;
        mbar_wait_u32(bfull(buf), (kb >> 1) & 1);
        tc_fence_after();
        const uint64_t db0 = kdesc(b_stage + buf * B_STAGE);
#pragma unroll
        for (int i = 0; i < S; i++, ause++) {
          const int slot = ause % A_SLOTS;
          mbar_wait_u32(afull(slot), (ause / A_SLOTS) & 1);
          tc_fence_after();
          const uint64_t da = kdesc(a_ring + slot * A_TILE);
#pragma unroll
          for (int j = 0; j < S - i; j++) {
            const uint64_t db = db0 + (uint64_t)((j * B_TILE) >> 4);
            const uint32_t dcol = tmem_d + (uint32_t)((i + j) * EN);
#pragma unroll
            for (int ks = 0; ks < EK / UK; ks++)
              tc_mma_i8(dcol, da + (uint64_t)((ks * UK) >> 4), db + (uint64_t)((ks * UK) >> 4), idesc, (kb == 0 && i == 0 && ks == 0) ? 0u : 1u, leader);
          }
          tc_commit_pred(aempty(slot), leader);
        }
        tc_commit_pred(bempty(buf), leader);
      }
      tc_commit_pred(tfull, leader);
    }
  } else {
    // ---- epilogue: warp w may only touch TMEM lanes 32 (w % 4) .. 32 (w % 4) + 31
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    if (nk > 0) {
      mbar_wait_u32(tfull, 0);
      tc_fence_after();
    }
#pragma unroll 1
    for (int half = 0; half < EN / 32; half++) {
      double v[32];
#pragma unroll
      for (int j = 0; j < 32; j++) v[j] = 0.0;
      if (nk > 0) {
        double w = 1.0;
#pragma unroll 1
        for (int gi = 0; gi < S; gi++, w *= (1.0 / 128.0)) {
          int r[32];
          tc_ld32_i(tmem_d + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(gi * EN + half * 32), r);
#pragma unroll
          for (int j = 0; j < 32; j++) v[j] = fma((double)r[j], w, v[j]);
        }
      }
      epi(tile_m, tile_n, z, row, half * 32, v);
    }
    tc_fence_before();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_d), "r"((uint32_t)TMEM_COLS) : "memory");
  }
}

// ---- host side: 3-D tensor map over slice planes [S][rows][ldk] of int8 (k contiguous); box = 128 k x box_rows rows x 1 slice ----------
inline bool make_map3(CUtensorMap* map, const signed char* ptr, uint64_t k, uint64_t rows, uint64_t ldk, uint64_t plane_bytes, uint32_t box_rows, int nslices = S) {
  t5::EncodeTiledFn fn = t5::encode_tiled_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {k, rows, (cuuint64_t)nslices};
  cuuint64_t strides[2] = {ldk, plane_bytes};
  cuuint32_t box[3] = {128, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// slices of a row-major FP64 matrix [rows][ld] (k contiguous): one warp per row -- row maximum, power-of-two scale, S planes [S][rows][ldk]
template <int NS = S>
__global__ void __launch_bounds__(256) slice_rows_kernel(const double* __restrict__ in, int64_t ld, int rows, int k, signed char* __restrict__ planes, int64_t ldk,
                                                         int64_t plane_bytes, double* __restrict__ scale) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const double* src = in + (int64_t)row * ld;
  double mx = 0.0;
  for (int c = lane; c < k; c += 32) mx = fmax(mx, fabs(src[c]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const double sc = pow2_scale(mx), inv = 1.0 / sc;
  if (lane == 0) scale[row] = sc;
  for (int c = lane; c < (int)ldk; c += 32) {
    signed char q[NS];
    slice_n<NS>(c < k ? src[c] : 0.0, inv, q);
#pragma unroll
    for (int i = 0; i < NS; i++) planes[i * plane_bytes + (int64_t)row * ldk + c] = q[i];
  }
}

// slices of the COLUMNS of a row-major FP64 matrix [rows][ld] (rows = k, columns = points), written point-major: planes [NS][cols][ldk] with
// k contiguous, one power-of-two scale per point from the exact column maximum.  One CTA per 32 points: a first pass over the strip for the
// maxima, a second one (an L2 hit: 32 x rows x 8 bytes) through a 32 x 32 shared-memory tile for the transposed, sliced stores.
// colmax != nullptr: the column maxima are already known (the producing epilogue tracked them with atomicMax) and the first pass is skipped.
template <int NS>
__global__ void __launch_bounds__(256) transpose_slice_kernel(const double* __restrict__ in, int64_t ld, int rows, int cols, signed char* __restrict__ planes,
                                                              int64_t ldk, int64_t plane_bytes, double* __restrict__ scale, const double* __restrict__ colmax = nullptr) {
  __shared__ double tile[32][33];
  __shared__ double smx[8][32];
  __shared__ double sinv[32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n0 = blockIdx.x * 32;
  const bool cok = n0 + tx < cols;
  double mx = 0.0;
  if (colmax) {
    if (ty == 0 && cok) mx = colmax[n0 + tx];
  } else {
    for (int r = ty; r < rows; r += 8) mx = fmax(mx, cok ? fabs(in[(int64_t)r * ld + n0 + tx]) : 0.0);
  }
  smx[ty][tx] = mx;
  __syncthreads();
  if (ty == 0) {
#pragma unroll
    for (int j = 1; j < 8; j++) mx = fmax(mx, smx[j][tx]);
    const double sc = pow2_scale(mx);
    if (cok) scale[n0 + tx] = sc;
    sinv[tx] = 1.0 / sc;
  }
  for (int r0 = 0; r0 < (int)ldk; r0 += 32) {
    __syncthreads();  // (also publishes sinv on the first pass)
    for (int j = ty; j < 32; j += 8) tile[j][tx] = (cok && r0 + j < rows) ? in[(int64_t)(r0 + j) * ld + n0 + tx] : 0.0;
    __syncthreads();
    // thread -> point ty * 4 + (tx >> 3), rows 4 (tx & 7) .. + 3: a warp stores 4 x 32 contiguous bytes per plane
    const int n = ty * 4 + (tx >> 3), r4 = (tx & 7) * 4;
    if (n0 + n < cols) {
      const double inv = sinv[n];
      signed char q[4][NS];
#pragma unroll
      for (int e = 0; e < 4; e++) slice_n<NS>(tile[r4 + e][n], inv, q[e]);
#pragma unroll
      for (int i = 0; i < NS; i++) {
        const char4 v = make_char4(q[0][i], q[1][i], q[2][i], q[3][i]);
        *reinterpret_cast<char4*>(planes + i * plane_bytes + (int64_t)(n0 + n) * ldk + r0 + r4) = v;
      }
    }
  }
}

// ---- operands of the Float64 mode's S6 (G += As A^T, k = the points of a launch group) ----------------------------------------------------
// The matrices are [rows = inducing index][ld] with the points contiguous, i.e. already K-major; what slice_rows_kernel (one warp per row) cannot do
// is a row of 1.5e5 points.  rowmax_kernel: grid (column segments, rows / 8), one warp per (row, segment), the maxima combined with atomicMax on
// the bit patterns (non-negative doubles order like their bits).  slice_rows2d_kernel: grid (column blocks of 1024, rows), four consecutive
// points per thread (char4 stores), scale from the finished row maximum; columns [k, ldk) are zero-filled.
__global__ void __launch_bounds__(256) rowmax_kernel(const double* __restrict__ in, int64_t ld, int rows, int k, int seg, unsigned long long* __restrict__ mx) {
  const int row = blockIdx.y * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int c0 = blockIdx.x * seg, c1 = min(k, c0 + seg);
  const double* src = in + (int64_t)row * ld;
  double m = 0.0;
  for (int c = c0 + lane; c < c1; c += 32) m = fmax(m, fabs(src[c]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) atomicMax(mx + row, (unsigned long long)__double_as_longlong(m));
}
template <int NS>
__global__ void __launch_bounds__(256) slice_rows2d_kernel(const double* __restrict__ in, int64_t ld, int k, signed char* __restrict__ planes, int64_t ldk,
                                                           int64_t plane_bytes, const unsigned long long* __restrict__ mx, double* __restrict__ scale) {
  const int row = blockIdx.y;
  const int c = (blockIdx.x * 256 + threadIdx.x) * 4;
  const double sc = 2.0 * pow2_scale(__longlong_as_double((long long)mx[row])), inv = 1.0 / sc;  // |x| / sc <= 1/2 (slice_rn)
  if (blockIdx.x == 0 && threadIdx.x == 0) scale[row] = sc;
  if (c >= (int)ldk) return;
  const double* src = in + (int64_t)row * ld;
  signed char q[4][NS];
#pragma unroll
  for (int e = 0; e < 4; e++) slice_rn<NS>(c + e < k ? src[c + e] : 0.0, inv, q[e]);
#pragma unroll
  for (int i = 0; i < NS; i++) *reinterpret_cast<char4*>(planes + i * plane_bytes + (int64_t)row * ldk + c) = make_char4(q[0][i], q[1][i], q[2][i], q[3][i]);
}
// G[z][row + col * Mp] += 2^-14 sA[row] sB[col] v   (A operand = As planes, B operand = A planes; lower tiles only; one slab of points per z)
struct EpiE6 {
  double* G;  // [nz][Mp * Mp], column-major slabs
  int Mp;
  const double* sA;
  const double* sB;
  __device__ __forceinline__ void operator()(int tm, int tn, int z, int row, int c0, const double (&v)[32]) const {
    const int r = tm * EM + row;
    const double f = sA[r] * (1.0 / 16384.0);
    double* p = G + (int64_t)z * Mp * Mp + (int64_t)(tn * EN + c0) * Mp + r;
    const double* sb = sB + tn * EN + c0;
#pragma unroll
    for (int j = 0; j < 32; j++) p[(int64_t)j * Mp] += v[j] * (f * sb[j]);
  }
};

}  // namespace i8e
}  // namespace agp
