// agp.cu -- host orchestration and the C ABI (include/agp.h) of the B200 SVGP / Laplace hot path.
//
// One translation unit: the device code lives in the headers included below.  Build:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC \
//        -o libagp_b200.so agp.cu -ldl
// The library links neither torch nor cuBLAS/cuSOLVER; NCCL is dlopen'ed on agp_comm_init.
#include <dlfcn.h>
#include <nccl.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/agp.h"
#include "dense.cuh"
#include "f32sweep.cuh"
#include "gemm.cuh"
#include "kfun.cuh"
#include "laplace.cuh"
#include "sweep.cuh"

using namespace agp;

// ---------------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static thread_local int32_t g_err_info = 0;  // PosDefException(info): the failing column of the last AGP_ERR_NOT_PD
static int32_t fail(int32_t code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CU(x)                                                                                        \
  do {                                                                                               \
    cudaError_t e_ = (x);                                                                            \
    if (e_ != cudaSuccess) return fail(AGP_ERR_CUDA, "%s failed: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)
#define OK(x)                      \
  do {                             \
    int32_t s_ = (x);              \
    if (s_ != AGP_OK) return s_;   \
  } while (0)

static int32_t fail_not_pd(const char* what, int column) {
  g_err_info = column;
  return fail(AGP_ERR_NOT_PD, "PosDefException: %s is not positive definite; Cholesky failed at column %d", what, column);
}
extern "C" const char* agp_last_error_string(void) { return g_err.c_str(); }
extern "C" int32_t agp_last_error_info(void) { return g_err_info; }
extern "C" int32_t agp_build_arch(void) { return 100; }

static inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }

// ---------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------
struct DevBuf {
  double* p = nullptr;
  int64_t n = 0;
  int32_t ensure(int64_t need) {
    if (need <= n) return AGP_OK;
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
    cudaError_t e = cudaMalloc(&p, sizeof(double) * need);
    if (e != cudaSuccess) return fail(AGP_ERR_ALLOC, "cudaMalloc of %lld doubles failed: %s", (long long)need, cudaGetErrorString(e));
    n = need;
    return AGP_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
};

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;
static int32_t load_nccl() {
  if (g_nccl.lib) return AGP_OK;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  if (!g_nccl.lib) return fail(AGP_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(g_nccl.lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(g_nccl.lib, "ncclCommInitRank");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(g_nccl.lib, "ncclAllReduce");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(g_nccl.lib, "ncclCommDestroy");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(g_nccl.lib, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy)
    return fail(AGP_ERR_NCCL, "libnccl is missing a required symbol");
  return AGP_OK;
}

// The INT8 products of S1 (Float32 mode) and of S2 / S6 (AGP_COMPUTE_F64_EMU) run from M = 768: at M = 512 the DMMA stages are as fast
// (C2 per step: 11.5 against 12.0 ms for S1, 10.7 against 11.3 ms for S6), while the INT8 S6 takes C4 350 -> 250 ms, C5 minibatch 139 -> 74 ms.
constexpr int I8_MIN_ROWS = 768;
// The emulated S2 / S6 run only on launch groups of at least this many points; narrower groups stay on DMMA.
constexpr int I8_MIN_COLS = 2048;

// Engine of each GEMM-shaped stage of the sweep, fixed per step by compute_dtype and M (resolve_params).
//   DMMA: the Float64 kernels of sweep.cuh / gemm.cuh (S1: kuf_gen_kernel + blocked TRSM);
//   TF32: 3xTF32 products on tcgen05 (f32sweep.cuh);  I8: FP64-accurate INT8-slice products on tcgen05 (i8emu.cuh; S5: five slices).
enum Engine { ENG_DMMA, ENG_TF32, ENG_I8 };
struct SweepPlan {
  int pts_tile = BN;  // launch groups are padded to this many points (128 in the tcgen05 modes)
  Engine s1 = ENG_DMMA, s2 = ENG_DMMA, s4 = ENG_DMMA, s5 = ENG_DMMA, s6 = ENG_DMMA;
  bool s7_streamed = false;  // S7 reads Kuf and kappa' back from S1 (plain stationary kinds) instead of recomputing them
  // the plan of one launch group of ncols points
  SweepPlan at_width(int ncols) const {
    SweepPlan g = *this;
    if (ncols < I8_MIN_COLS) {
      if (g.s2 == ENG_I8) g.s2 = ENG_DMMA;
      if (g.s6 == ENG_I8) g.s6 = ENG_DMMA;
    }
    return g;
  }
};

// Everything the sweep needs that depends on one agp_svgp_params (uploaded once per step).
struct SvgpState {
  bool valid = false;
  bool sweep_pending = false;  // agp_svgp_sweep has filled the reduce buffer and agp_svgp_finish has not consumed it yet
  SweepPlan plan;
  int M = 0, Mp = 0, D = 0, nb = 0;
  int n_scale = 1;
  bool centered = false;
  double mean_const = 0, jitter = 0, scale = 1;
  int want_grad = 0;
  long long point_base = 0;  // Monte-Carlo counter offset of the batch being swept (dataset offset + rank shard offset)
  KernelParams kp;
  LikParams lp;
  std::vector<double> h_m;  // padded host copy of m
};

// Optional per-kernel-class timing with CUDA events on the context's stream (agp_ctx_profile*):
// this is how bench.py measures the launch durations behind its roofline figures.
enum { PC_TRSM_FWD = 0, PC_GEMM_BTA, PC_PERPOINT, PC_GEMM_BC, PC_TRSM_BWD, PC_SYRK, PC_KGRAD, PC_PREPARE, PC_FINISH, PC_ALLREDUCE, PC_LAPLACE, PC_F32_AUX, PC_COUNT };
static const char* const kProfNames[PC_COUNT] = {"trsm_kuf_fwd", "gemm_BtA", "perpoint", "gemm_BC", "trsm_bwd", "syrk_G", "kgrad",
                                                 "prepare_step", "finish_epilogue", "allreduce", "laplace", "f32_planes_gvec"};
struct ProfRec {
  int cls;
  cudaEvent_t a, b;
};
struct Prof {
  bool on = false;
  std::vector<cudaEvent_t> pool;
  size_t used = 0;
  std::vector<ProfRec> recs;
  double ms[PC_COUNT] = {0};
  int64_t cnt[PC_COUNT] = {0};
  cudaEvent_t get() {
    if (used == pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      pool.push_back(e);
    }
    return pool[used++];
  }
};

static void lap_release(agp_ctx* c);
static void chol_partition_release(agp_ctx* c);
struct agp_ctx {
  Prof prof;
  void* lap = nullptr;  // LapWork (laplace_host.inc)
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;                // trailing updates of the blocked Cholesky (look-ahead), see blocked_cholesky
  cudaEvent_t ev_trail = nullptr;
  cudaStream_t stream3 = nullptr;                // tile-level look-ahead of the blocked Cholesky: full-height panels / in-super-panel updates
  // SM partition for large factorisations (green contexts, see chol_partition): the critical chain on its own 8 SMs
  int part_state = 0;                            // 0 = not tried, 1 = in use, -1 = unavailable
  CUgreenCtx part_chain = nullptr, part_bulk = nullptr;
  cudaStream_t pstream_chain = nullptr, pstream_side = nullptr, pstream_trail = nullptr;
  cudaEvent_t ev_enter = nullptr, ev_leave = nullptr;
  int part_sms_chain = 0, part_sms_bulk = 0;
  cudaEvent_t ev_diag = nullptr, ev_prow = nullptr, ev_side = nullptr, ev_prio = nullptr;
  cudaStream_t stream_copy = nullptr;            // upload of the q.Sigma factor (M^2 doubles) behind the Kuu factorisation, see prepare_step
  cudaEvent_t ev_copy = nullptr;
  int sms = 148;
  int64_t launches = 0;
  int64_t chunk_cols = 0;  // capacity of the per-chunk scratch (columns)
  int nslab = 0, nsplit = 0;
  // once-per-step M x M operands (column-major, ld = Mp unless noted)
  DevBuf z, zs, zn, zsp, mvec, mt, Lq, Kw, Lk, Lt, Ut, Bt_cm, Bt_rm, W1, W2, W3, W4, vec64, vec64b;
  // per-chunk scratch [Mp][chunk_cols]
  DevBuf A, C, Ab, As, saa, sam, scc_part, dmu, dv, sc_part;
  DevBuf Kf, DKb;  // reverse pass, stationary kernels: Kuf and variance * kappa'(u) of the launch group, kept from S1 for S7
  // accumulators
  DevBuf gpart, Gpart, kpart, red, small, ghbuf;
  DevBuf qBt7, sBt7, sPm;  // AGP_COMPUTE_F64_EMU, S2: slices / scales of Bt^T (once per sweep), per-point scales of the point-major slices of A
  DevBuf q6A, q6As, s6;  // AGP_COMPUTE_F64_EMU, S6 on the INT8 tensor path: slice planes of A and As, [scales A | scales As | row maxima x 2]
  // Float32 mode: hi | lo FP32 planes (each DevBuf holds both: 2 x count floats = count doubles)
  DevBuf fA, fC, fAb, fAs, fBtc, fBtr, fLi;
  DevBuf qAb, sAb, qLi, sLi;
  DevBuf qK, sK, qLi7, sLi7, sxx_part;  // Float32 mode, forward solve on the INT8 tensor path: 7 slice planes of Kuf (point-major) and of Linv, scales, column-sum partials  // Float32 mode, S5 on the INT8 tensor path: 4 slice planes of Ab (point-major) and of Linv^T, their scales
  int* d_flags = nullptr;  // [0] potrf info, [1] domain flag
  SvgpState st;
  ncclComm_t comm = nullptr;
  int nranks = 1, rank = 0;
  // prediction outputs / scratch
  DevBuf mu_out, var_out, px1, px2, pxs1, pxn1, pxs2, pxn2, pcov;
};

struct agp_dataset {
  agp_ctx* ctx = nullptr;
  int64_t cap = 0, N = 0;
  int D = 0;
  double* X = nullptr;  // point-major [cap][D]
  double* y = nullptr;
  DevBuf stage;
};

#define LAUNCHED(ctx) ((ctx)->launches++)
struct ProfScope {
  agp_ctx* c;
  bool on;
  ProfScope(agp_ctx* c_, int cls) : c(c_), on(c_->prof.on) {
    if (!on) return;
    ProfRec r{cls, c->prof.get(), c->prof.get()};
    cudaEventRecord(r.a, c->stream);
    c->prof.recs.push_back(r);
  }
  ~ProfScope() {
    if (on) cudaEventRecord(c->prof.recs.back().b, c->stream);
  }
};
#define KCHECK()                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = cudaGetLastError();                                                           \
    if (e_ != cudaSuccess) return fail(AGP_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

extern "C" int32_t agp_ctx_create(int32_t device, agp_ctx** out) {
  if (!out) return fail(AGP_ERR_INVALID, "agp_ctx_create: out is NULL");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(AGP_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(AGP_ERR_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return fail(AGP_ERR_UNSUPPORTED, "device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
  agp_ctx* c = new agp_ctx();
  c->device = device;
  c->sms = prop.multiProcessorCount;
  // the main stream outranks the look-ahead stream: the latency-bound chain of the blocked Cholesky must get the first CTA
  // slot that the trailing update frees (blocked_cholesky)
  int prio_lo = 0, prio_hi = 0;
  CU(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  CU(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_hi));
  CU(cudaStreamCreateWithPriority(&c->stream2, cudaStreamNonBlocking, prio_lo));
  CU(cudaStreamCreateWithPriority(&c->stream3, cudaStreamNonBlocking, prio_hi < prio_lo - 1 ? prio_hi + 1 : prio_hi));
  CU(cudaEventCreateWithFlags(&c->ev_trail, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_diag, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_prow, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_side, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_prio, cudaEventDisableTiming));
  CU(cudaStreamCreateWithFlags(&c->stream_copy, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&c->ev_copy, cudaEventDisableTiming));
  CU(cudaMalloc(&c->d_flags, 4 * sizeof(int)));
  CU(cudaMemset(c->d_flags, 0, 4 * sizeof(int)));
  *out = c;
  return AGP_OK;
}

extern "C" int32_t agp_ctx_destroy(agp_ctx* c) {
  if (!c) return AGP_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
  DevBuf* bufs[] = {&c->z, &c->zs, &c->zn, &c->zsp, &c->mvec, &c->mt, &c->Lq, &c->Kw, &c->Lk, &c->Lt, &c->Ut, &c->Bt_cm, &c->Bt_rm,
                    &c->W1, &c->W2, &c->W3, &c->W4, &c->vec64, &c->vec64b, &c->A, &c->C, &c->Ab, &c->As, &c->Kf, &c->DKb, &c->saa, &c->sam,
                    &c->scc_part, &c->dmu, &c->dv, &c->sc_part, &c->gpart, &c->Gpart, &c->kpart, &c->red, &c->small, &c->ghbuf, &c->q6A, &c->q6As, &c->s6, &c->qBt7, &c->sBt7, &c->sPm, &c->fA, &c->fC, &c->fAb, &c->fAs, &c->fBtc, &c->fBtr, &c->fLi, &c->qAb, &c->sAb, &c->qLi, &c->sLi, &c->qK, &c->sK, &c->qLi7, &c->sLi7, &c->sxx_part,
                    &c->mu_out, &c->var_out, &c->px1, &c->px2, &c->pxs1, &c->pxn1, &c->pxs2, &c->pxn2, &c->pcov};
  for (DevBuf* b : bufs) b->release();
  lap_release(c);
  if (c->d_flags) cudaFree(c->d_flags);
  for (cudaEvent_t e : c->prof.pool) cudaEventDestroy(e);
  if (c->ev_trail) cudaEventDestroy(c->ev_trail);
  if (c->stream2) cudaStreamDestroy(c->stream2);
  for (cudaEvent_t e : {c->ev_diag, c->ev_prow, c->ev_side, c->ev_prio})
    if (e) cudaEventDestroy(e);
  if (c->stream3) cudaStreamDestroy(c->stream3);
  chol_partition_release(c);
  if (c->ev_copy) cudaEventDestroy(c->ev_copy);
  if (c->stream_copy) cudaStreamDestroy(c->stream_copy);
  cudaStreamDestroy(c->stream);
  delete c;
  return AGP_OK;
}

extern "C" int32_t agp_ctx_stream(agp_ctx* c, void** s) {
  if (!c || !s) return fail(AGP_ERR_INVALID, "agp_ctx_stream: NULL argument");
  *s = (void*)c->stream;
  return AGP_OK;
}
extern "C" int32_t agp_ctx_profile(agp_ctx* c, int32_t enable) {
  if (!c) return fail(AGP_ERR_INVALID, "agp_ctx_profile: NULL");
  c->prof.on = enable != 0;
  return AGP_OK;
}
extern "C" const char* agp_profile_class_name(int32_t cls) { return (cls >= 0 && cls < PC_COUNT) ? kProfNames[cls] : nullptr; }
extern "C" int32_t agp_ctx_profile_read(agp_ctx* c, int32_t max_classes, double* ms_out, int64_t* count_out, int32_t* n_classes) {
  if (!c) return fail(AGP_ERR_INVALID, "agp_ctx_profile_read: NULL");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  Prof& p = c->prof;
  for (const ProfRec& r : p.recs) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      p.ms[r.cls] += ms;
      p.cnt[r.cls]++;
    }
  }
  p.recs.clear();
  p.used = 0;
  for (int i = 0; i < PC_COUNT && i < max_classes; i++) {
    if (ms_out) ms_out[i] = p.ms[i];
    if (count_out) count_out[i] = p.cnt[i];
  }
  if (n_classes) *n_classes = PC_COUNT;
  for (int i = 0; i < PC_COUNT; i++) {
    p.ms[i] = 0;
    p.cnt[i] = 0;
  }
  return AGP_OK;
}
extern "C" int32_t agp_ctx_launch_count(agp_ctx* c, int64_t* out) {
  if (!c || !out) return fail(AGP_ERR_INVALID, "agp_ctx_launch_count: NULL argument");
  *out = c->launches;
  return AGP_OK;
}

// ---------------------------------------------------------------------------------------------------
// communicator
// ---------------------------------------------------------------------------------------------------
extern "C" int32_t agp_comm_unique_id(void* id128) {
  if (!id128) return fail(AGP_ERR_INVALID, "agp_comm_unique_id: NULL");
  OK(load_nccl());
  ncclUniqueId id;
  ncclResult_t r = g_nccl.GetUniqueId(&id);
  if (r != ncclSuccess) return fail(AGP_ERR_NCCL, "ncclGetUniqueId: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  memcpy(id128, &id, 128);
  return AGP_OK;
}
extern "C" int32_t agp_comm_init(agp_ctx* c, int32_t nranks, int32_t rank, const void* id128) {
  if (!c || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(AGP_ERR_INVALID, "agp_comm_init: bad arguments");
  OK(load_nccl());
  CU(cudaSetDevice(c->device));
  ncclUniqueId id;
  memcpy(&id, id128, 128);
  ncclResult_t r = g_nccl.CommInitRank(&c->comm, nranks, id, rank);
  if (r != ncclSuccess) return fail(AGP_ERR_NCCL, "ncclCommInitRank: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  c->nranks = nranks;
  c->rank = rank;
  return AGP_OK;
}
extern "C" int32_t agp_comm_destroy(agp_ctx* c) {
  if (c && c->comm) {
    g_nccl.CommDestroy(c->comm);
    c->comm = nullptr;
    c->nranks = 1;
    c->rank = 0;
  }
  return AGP_OK;
}

// ---------------------------------------------------------------------------------------------------
// datasets
// ---------------------------------------------------------------------------------------------------
__global__ void feature_to_point_major_kernel(const double* in, int64_t ldx, double* out, int64_t N, int D) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N * D; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / D;
    const int d = (int)(i % D);
    out[i] = in[(int64_t)d * ldx + n];
  }
}
template <typename T>
__global__ void convert_y_kernel(const T* in, double* out, int64_t N) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) out[i] = (double)in[i];
}

extern "C" int32_t agp_dataset_create(agp_ctx* c, int64_t capacity, int32_t D, agp_dataset** out) {
  if (!c || !out || capacity < 1 || D < 1) return fail(AGP_ERR_INVALID, "agp_dataset_create: bad arguments");
  if (D > MAXD) return fail(AGP_ERR_UNSUPPORTED, "input dimension %d > %d is not supported on device", D, MAXD);
  CU(cudaSetDevice(c->device));
  agp_dataset* ds = new agp_dataset();
  ds->ctx = c;
  ds->cap = capacity;
  ds->D = D;
  // one tile of slack so a partially filled last column tile can be staged without reading out of bounds
  cudaError_t e = cudaMalloc(&ds->X, sizeof(double) * (capacity + BN) * D);
  if (e == cudaSuccess) e = cudaMalloc(&ds->y, sizeof(double) * (capacity + BN));
  if (e != cudaSuccess) {
    delete ds;
    return fail(AGP_ERR_ALLOC, "dataset allocation failed: %s", cudaGetErrorString(e));
  }
  *out = ds;
  return AGP_OK;
}

// observations: F64 as is, F32 / I64 / U8 (Bool) widened on the device
static int32_t upload_y(agp_dataset* ds, const void* y, int64_t N, int32_t ytype, int32_t location) {
  agp_ctx* c = ds->ctx;
  const cudaMemcpyKind kind = location == AGP_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  if (y) {
    if (ytype == AGP_Y_F64) {
      CU(cudaMemcpyAsync(ds->y, y, sizeof(double) * N, kind, c->stream));
    } else {
      const size_t esz = ytype == AGP_Y_F32 ? 4 : ytype == AGP_Y_I64 ? 8 : ytype == AGP_Y_U8 ? 1 : 0;
      if (!esz) return fail(AGP_ERR_INVALID, "unknown ytype %d", ytype);
      const void* src = y;
      if (location == AGP_HOST) {
        OK(ds->stage.ensure((int64_t)((esz * N + 7) / 8) + 1));
        CU(cudaMemcpyAsync(ds->stage.p, y, esz * N, cudaMemcpyHostToDevice, c->stream));
        src = ds->stage.p;
      }
      if (ytype == AGP_Y_F32) convert_y_kernel<float><<<1024, 256, 0, c->stream>>>((const float*)src, ds->y, N);
      if (ytype == AGP_Y_I64) convert_y_kernel<long long><<<1024, 256, 0, c->stream>>>((const long long*)src, ds->y, N);
      if (ytype == AGP_Y_U8) convert_y_kernel<unsigned char><<<1024, 256, 0, c->stream>>>((const unsigned char*)src, ds->y, N);
      LAUNCHED(c);
      KCHECK();
    }
  }
  return AGP_OK;
}

extern "C" int32_t agp_dataset_upload(agp_dataset* ds, const void* X, int64_t N, int64_t ldx, int32_t layout, const void* y,
                                      int32_t ytype, int32_t location) {
  if (!ds || !X || N < 0 || N > ds->cap) return fail(AGP_ERR_INVALID, "agp_dataset_upload: bad arguments (N=%lld, cap=%lld)", (long long)N, ds ? (long long)ds->cap : -1LL);
  agp_ctx* c = ds->ctx;
  CU(cudaSetDevice(c->device));
  const int D = ds->D;
  const cudaMemcpyKind kind = location == AGP_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  if (layout == AGP_POINT_MAJOR) {
    if (ldx <= 0) ldx = D;
    if (ldx == D)
      CU(cudaMemcpyAsync(ds->X, X, sizeof(double) * N * D, kind, c->stream));
    else
      CU(cudaMemcpy2DAsync(ds->X, sizeof(double) * D, X, sizeof(double) * ldx, sizeof(double) * D, N, kind, c->stream));
  } else if (layout == AGP_FEATURE_MAJOR) {
    if (ldx <= 0) ldx = N;
    const double* src = (const double*)X;
    if (location == AGP_HOST) {
      OK(ds->stage.ensure(ldx * D));
      CU(cudaMemcpyAsync(ds->stage.p, X, sizeof(double) * ldx * D, cudaMemcpyHostToDevice, c->stream));
      src = ds->stage.p;
    }
    feature_to_point_major_kernel<<<1024, 256, 0, c->stream>>>(src, ldx, ds->X, N, D);
    LAUNCHED(c);
    KCHECK();
  } else {
    return fail(AGP_ERR_INVALID, "unknown layout %d", layout);
  }
  OK(upload_y(ds, y, N, ytype, location));
  CU(cudaStreamSynchronize(c->stream));
  ds->N = N;
  return AGP_OK;
}

// Float32 inputs (a Float32 caller's ColVecs / RowVecs): half the PCIe bytes; widened to the FP64 the kernels compute in.
__global__ void widen_x_kernel(const float* in, int64_t ldx, int layout, double* out, int64_t N, int D) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N * D; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / D;
    const int d = (int)(i % D);
    out[i] = (double)(layout == AGP_FEATURE_MAJOR ? in[(int64_t)d * ldx + n] : in[n * ldx + d]);
  }
}
extern "C" int32_t agp_dataset_upload_f32(agp_dataset* ds, const float* X, int64_t N, int64_t ldx, int32_t layout, const void* y,
                                          int32_t ytype, int32_t location) {
  if (!ds || !X || N < 0 || N > ds->cap) return fail(AGP_ERR_INVALID, "agp_dataset_upload_f32: bad arguments (N=%lld, cap=%lld)", (long long)N, ds ? (long long)ds->cap : -1LL);
  if (layout != AGP_POINT_MAJOR && layout != AGP_FEATURE_MAJOR) return fail(AGP_ERR_INVALID, "unknown layout %d", layout);
  agp_ctx* c = ds->ctx;
  CU(cudaSetDevice(c->device));
  const int D = ds->D;
  if (ldx <= 0) ldx = layout == AGP_POINT_MAJOR ? D : N;
  const int64_t nflt = layout == AGP_POINT_MAJOR ? N * ldx : (int64_t)D * ldx;
  const float* src = X;
  if (location == AGP_HOST && N > 0) {
    OK(ds->stage.ensure((nflt + 1) / 2 + 1));
    CU(cudaMemcpyAsync(ds->stage.p, X, sizeof(float) * nflt, cudaMemcpyHostToDevice, c->stream));
    src = reinterpret_cast<const float*>(ds->stage.p);
  }
  if (N > 0) {
    widen_x_kernel<<<1024, 256, 0, c->stream>>>(src, ldx, layout, ds->X, N, D);
    LAUNCHED(c);
    KCHECK();
  }
  CU(cudaStreamSynchronize(c->stream));  // the staging buffer is reused for the observations
  OK(upload_y(ds, y, N, ytype, location));
  CU(cudaStreamSynchronize(c->stream));
  ds->N = N;
  return AGP_OK;
}

extern "C" int32_t agp_dataset_size(agp_dataset* ds, int64_t* N, int32_t* D) {
  if (!ds) return fail(AGP_ERR_INVALID, "agp_dataset_size: NULL");
  if (N) *N = ds->N;
  if (D) *D = ds->D;
  return AGP_OK;
}
extern "C" int32_t agp_dataset_destroy(agp_dataset* ds) {
  if (!ds) return AGP_OK;
  cudaSetDevice(ds->ctx->device);
  if (ds->X) cudaFree(ds->X);
  if (ds->y) cudaFree(ds->y);
  ds->stage.release();
  delete ds;
  return AGP_OK;
}

// ---------------------------------------------------------------------------------------------------
// launch helpers
// ---------------------------------------------------------------------------------------------------
// Opt-in dynamic shared memory, set once per kernel instantiation and device (not on every launch: the call costs
// a few microseconds, which matters for the latency-bound small-M path).
template <auto Kernel>
static int32_t ensure_smem(agp_ctx* c, int bytes) {
  static int granted[64] = {0};
  int& g = granted[c->device & 63];
  if (g > bytes) return AGP_OK;  // g = granted bytes + 1
  if (bytes > 0) CU(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  g = bytes + 1;
  return AGP_OK;
}

template <int MODE, int S>
static int32_t launch_trsm_s(agp_ctx* c, const TrsmArgs& a, int tiles_n) {
  using Cfg = StageCfg<A_KM, B_KN>;
  const int Sx = MODE == TR_KUF_FWD_SCALED ? kuf_dp(a.kp.D) + 2 : 0;
  const int smem = (S * (Cfg::elems + BK * Sx) + 64 * Sx) * 8 + 16;
  OK((ensure_smem<trsm_kernel<MODE, S>>(c, smem)));
  trsm_kernel<MODE, S><<<tiles_n, NTHREADS, smem, c->stream>>>(a);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}
// 4 pipeline stages; the Kuf generator drops to 3 when the z slabs of a wide input (D > 8) would cost the second CTA per SM
template <int MODE>
static int32_t launch_trsm(agp_ctx* c, const TrsmArgs& a, int tiles_n) {
  if constexpr (MODE == TR_KUF_FWD_SCALED) {
    if (a.kp.D > 8) return launch_trsm_s<MODE, 3>(c, a, tiles_n);
  }
  return launch_trsm_s<MODE, 4>(c, a, tiles_n);
}

// S1 = cov(f.prior, z, x) + the forward solve (SVA.jl:216-217): kuf_gen_kernel writes the Kuf tile of the launch group into X and the
// solve runs in place on it (TR_RHS_FWD_SUMS), with the column sums a^T a and a^T mt.
// keep = true (reverse pass of a stationary kernel): Kuf goes to c->Kf and variance * kappa'(u) to c->DKb, the solve reads Kf and writes
// t1.X; S7 then contracts the cotangent with the stored values (kgrad_kernel FAST) instead of recomputing distances and exp.
// gen_only = true: only the generator runs (into c->Kf); the caller solves by other means (Float32 mode: INT8 product with the explicit inverse).
static int32_t launch_s1(agp_ctx* c, const TrsmArgs& t1_in, int tiles_n, bool keep = false, bool gen_only = false) {
  TrsmArgs t1 = t1_in;
  KufGenArgs g{};
  // (SqExponential: kappa' = -kappa / 2, S7 needs only Kuf itself: one matrix written here instead of two)
  g.K = keep ? c->Kf.p : t1.X;
  g.DK = (keep && t1.kp.kind != AGP_KERNEL_SE) ? c->DKb.p : nullptr;
  if (keep) t1.RHS = c->Kf.p;
  g.ldx = t1.ldx;
  g.ncols = tiles_n * BN;
  g.pts = t1.pts;
  g.npts = t1.npts;
  g.zsp = t1.zsp;
  g.kp = t1.kp;
  const int D = t1.kp.D;
  const int smem = 0;  // static: KG_ROWS x (DMAX + 2) doubles (34 KB at DMAX = 32)
  const dim3 grid((g.ncols + KG_COLS - 1) / KG_COLS, t1.nb * BM / KG_ROWS);
#define AGP_KGEN_D(KD)                                                                   \
  {                                                                                      \
    if (D <= 4) kuf_gen_kernel<4, KD><<<grid, KG_COLS, smem, c->stream>>>(g);            \
    else if (D <= 8) kuf_gen_kernel<8, KD><<<grid, KG_COLS, smem, c->stream>>>(g);       \
    else if (D <= 16) kuf_gen_kernel<16, KD><<<grid, KG_COLS, smem, c->stream>>>(g);     \
    else kuf_gen_kernel<32, KD><<<grid, KG_COLS, smem, c->stream>>>(g);                  \
  }
  switch (t1.kp.kind) {
    case AGP_KERNEL_SE: AGP_KGEN_D(AGP_KERNEL_SE) break;
    case AGP_KERNEL_MATERN32: AGP_KGEN_D(AGP_KERNEL_MATERN32) break;
    case AGP_KERNEL_MATERN52: AGP_KGEN_D(AGP_KERNEL_MATERN52) break;
    case AGP_KERNEL_LINEAR: AGP_KGEN_D(AGP_KERNEL_LINEAR) break;
    default: AGP_KGEN_D(AGP_KERNEL_SUM) break;
  }
#undef AGP_KGEN_D
  LAUNCHED(c);
  KCHECK();
  if (gen_only) return AGP_OK;
  return launch_trsm<TR_RHS_FWD_SUMS>(c, t1, tiles_n);
}

// X <- Lk^-1 X (TR_RHS_FWD) or Lk^-T X (TR_RHS_BWD) in place; X row-major [Mp][ldx], tiles_n tiles of 64 columns
template <int MODE>
static int32_t solve_lk(agp_ctx* c, double* X, int64_t ldx, int tiles_n) {
  TrsmArgs a{};
  a.T = MODE == TR_RHS_BWD ? c->Ut.p : c->Lt.p;
  a.ldt = c->st.Mp;
  a.nb = c->st.nb;
  a.X = X;
  a.ldx = ldx;
  a.kp = c->st.kp;
  return launch_trsm<MODE>(c, a, tiles_n);
}

template <int LA, int LB, int S = StageCfg<LA, LB>::stages, class Epi>
static int32_t run_gemm(agp_ctx* c, int tiles_m, int tiles_n, const double* A, int64_t lda, const double* B, int64_t ldb, int K,
                        int kmode, int tmode, const Epi& epi) {
  using Cfg = StageCfg<LA, LB>;
  constexpr int smem_bytes = S * Cfg::bytes;
  GemmArgs g{A, lda, B, ldb, K, kmode, tmode};
  OK((ensure_smem<gemm_kernel<LA, LB, Epi, S>>(c, smem_bytes)));
  dim3 grid(tiles_m, tiles_n);
  if ((kmode == KR_LOWER || kmode == KR_UPPER) && tmode == TS_ALL && tiles_m > 1) {
    g.swizzle = std::max(1, c->sms);  // half a wave of column tiles per super-group
    g.tiles_m = tiles_m;
    g.tiles_n = tiles_n;
    grid = dim3(tiles_m * tiles_n, 1);
  }
  gemm_kernel<LA, LB, Epi, S><<<grid, NTHREADS, smem_bytes, c->stream>>>(g, epi);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}

static EpiStore epi_store(double* C, int64_t ldc, bool rowmajor, double alpha = 1.0, double beta = 0.0, int mask = MASK_NONE,
                          double diag_add = 0.0, const double* u = nullptr, const double* v = nullptr, double r1 = 0.0) {
  EpiStore e;
  e.C = C;
  e.ldc = ldc;
  e.rowmajor = rowmajor ? 1 : 0;
  e.alpha = alpha;
  e.beta = beta;
  e.mask = mask;
  e.diag_add = diag_add;
  e.r1u = u;
  e.r1v = v;
  e.r1 = r1;
  return e;
}

static int32_t fill(agp_ctx* c, double* p, int64_t n, double v) {
  if (n <= 0) return AGP_OK;
  if (v == 0.0) {
    CU(cudaMemsetAsync(p, 0, sizeof(double) * n, c->stream));
    return AGP_OK;
  }
  fill_kernel<<<(int)std::min<int64_t>(1024, (n + 255) / 256), 256, 0, c->stream>>>(p, n, v);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}

static int32_t transpose(agp_ctx* c, const double* in, double* out, int n, int64_t ld) {
  dim3 grid(n / 32, n / 32), block(32, 8);
  transpose_kernel<<<grid, block, 0, c->stream>>>(in, out, n, ld);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}

// launch helpers use c->stream: point it at another stream for a scope
struct StreamSwap {
  agp_ctx* c;
  cudaStream_t saved;
  StreamSwap(agp_ctx* c_, cudaStream_t s) : c(c_), saved(c_->stream) { c->stream = s; }
  ~StreamSwap() { c->stream = saved; }
};

// ---- SM partition for the blocked Cholesky (CUDA green contexts) ---------------------------------------------------------
// The chain of a large factorisation (diagonal-block kernel -> block row of the panel -> tile update -> next diagonal block) is a
// sequence of one-CTA / sixteen-CTA launches whose latency is the critical path once few block rows are left.  Stream priorities give
// those CTAs the first free slot, but not a quiet SM: next to a DMMA tile of the trailing update, which keeps the FP64 pipe of its SM
// busy, the one-warp column loop of the diagonal kernel runs 1.5-3x slower (80 -> 120..270 us, profiles/r3i_chol_trace_v2.txt).  So
// for nb >= 32 the device is split: 8 SMs (the smallest partition sm_100 allows) carry only the chain, the other 140 carry
// the panel / update / trailing GEMMs.  Streams of the two green contexts synchronise through events like any others; the rest of the
// library keeps using the primary context's streams (all 148 SMs).  If the driver refuses any step, the unpartitioned schedule is used.
struct GreenApi {
  CUresult (*DeviceGet)(CUdevice*, int) = nullptr;
  CUresult (*DeviceGetDevResource)(CUdevice, CUdevResource*, CUdevResourceType) = nullptr;
  CUresult (*DevSmResourceSplitByCount)(CUdevResource*, unsigned int*, const CUdevResource*, CUdevResource*, unsigned int, unsigned int) = nullptr;
  CUresult (*DevResourceGenerateDesc)(CUdevResourceDesc*, CUdevResource*, unsigned int) = nullptr;
  CUresult (*GreenCtxCreate)(CUgreenCtx*, CUdevResourceDesc, CUdevice, unsigned int) = nullptr;
  CUresult (*GreenCtxDestroy)(CUgreenCtx) = nullptr;
  CUresult (*GreenCtxStreamCreate)(CUstream*, CUgreenCtx, unsigned int, int) = nullptr;
  bool ok = false;
};
static GreenApi& green_api() {
  static GreenApi g;
  static bool tried = false;
  if (tried) return g;
  tried = true;
  auto get = [](const char* name, void** fn) {
    cudaDriverEntryPointQueryResult q;
    return cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess && *fn;
  };
  g.ok = get("cuDeviceGet", (void**)&g.DeviceGet) && get("cuDeviceGetDevResource", (void**)&g.DeviceGetDevResource) &&
         get("cuDevSmResourceSplitByCount", (void**)&g.DevSmResourceSplitByCount) && get("cuDevResourceGenerateDesc", (void**)&g.DevResourceGenerateDesc) &&
         get("cuGreenCtxCreate", (void**)&g.GreenCtxCreate) && get("cuGreenCtxDestroy", (void**)&g.GreenCtxDestroy) &&
         get("cuGreenCtxStreamCreate", (void**)&g.GreenCtxStreamCreate);
  return g;
}
static bool chol_partition(agp_ctx* c) {
  if (c->part_state != 0) return c->part_state > 0;
  c->part_state = -1;
  if (getenv("AGP_CHOL_PARTITION") && atoi(getenv("AGP_CHOL_PARTITION")) == 0) return false;  // for profilers that cannot follow green-context streams
  GreenApi& g = green_api();
  if (!g.ok) return false;
  CUdevice dev;
  CUdevResource all, grp[1], rest;
  unsigned int ngrp = 1;
  CUdevResourceDesc d_chain, d_bulk;
  if (g.DeviceGet(&dev, c->device) != CUDA_SUCCESS) return false;
  if (g.DeviceGetDevResource(dev, &all, CU_DEV_RESOURCE_TYPE_SM) != CUDA_SUCCESS) return false;
  if (g.DevSmResourceSplitByCount(grp, &ngrp, &all, &rest, 0, 8) != CUDA_SUCCESS || ngrp < 1) return false;
  if (grp[0].sm.smCount < 4 || rest.sm.smCount < all.sm.smCount / 2) return false;
  if (g.DevResourceGenerateDesc(&d_chain, &grp[0], 1) != CUDA_SUCCESS || g.DevResourceGenerateDesc(&d_bulk, &rest, 1) != CUDA_SUCCESS) return false;
  if (g.GreenCtxCreate(&c->part_chain, d_chain, dev, CU_GREEN_CTX_DEFAULT_STREAM) != CUDA_SUCCESS) return false;
  if (g.GreenCtxCreate(&c->part_bulk, d_bulk, dev, CU_GREEN_CTX_DEFAULT_STREAM) != CUDA_SUCCESS) {
    chol_partition_release(c);
    return false;
  }
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  CUstream s1 = nullptr, s2 = nullptr, s3 = nullptr;
  if (g.GreenCtxStreamCreate(&s1, c->part_chain, CU_STREAM_NON_BLOCKING, prio_hi) != CUDA_SUCCESS ||
      g.GreenCtxStreamCreate(&s2, c->part_bulk, CU_STREAM_NON_BLOCKING, prio_hi) != CUDA_SUCCESS ||
      g.GreenCtxStreamCreate(&s3, c->part_bulk, CU_STREAM_NON_BLOCKING, prio_lo) != CUDA_SUCCESS ||
      cudaEventCreateWithFlags(&c->ev_enter, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_leave, cudaEventDisableTiming) != cudaSuccess) {
    c->pstream_chain = (cudaStream_t)s1;
    c->pstream_side = (cudaStream_t)s2;
    c->pstream_trail = (cudaStream_t)s3;
    chol_partition_release(c);
    cudaGetLastError();
    return false;
  }
  c->pstream_chain = (cudaStream_t)s1;
  c->pstream_side = (cudaStream_t)s2;
  c->pstream_trail = (cudaStream_t)s3;
  c->part_sms_chain = (int)grp[0].sm.smCount;
  c->part_sms_bulk = (int)rest.sm.smCount;
  c->part_state = 1;
  if (getenv("AGP_CHOL_TRACE")) fprintf(stderr, "[chol partition] chain %d SMs, GEMMs %d SMs\n", c->part_sms_chain, c->part_sms_bulk);
  return true;
}
static void chol_partition_release(agp_ctx* c) {
  for (cudaStream_t* st : {&c->pstream_chain, &c->pstream_side, &c->pstream_trail})
    if (*st) {
      cudaStreamSynchronize(*st);
      cudaStreamDestroy(*st);
      *st = nullptr;
    }
  for (cudaEvent_t* e : {&c->ev_enter, &c->ev_leave})
    if (*e) {
      cudaEventDestroy(*e);
      *e = nullptr;
    }
  GreenApi& g = green_api();
  for (CUgreenCtx* gc : {&c->part_chain, &c->part_bulk})
    if (*gc) {
      if (g.GreenCtxDestroy) g.GreenCtxDestroy(*gc);
      *gc = nullptr;
    }
  c->part_state = -1;
}

// Two-level blocked right-looking Cholesky of the n x n (n = nb*128) matrix Kw (column-major, lower triangle read,
// destroyed) into L; also produces the inverse diagonal blocks in the diagonal blocks of Lt (inv) and Ut (inv^T).
// Inner level: 128-blocks (diagonal kernel + panel GEMM + an update confined to the current 512-wide super-panel);
// outer level: one trailing update per super-panel with K = 512, which quadruples the flop per byte of the
// dominant GEMM compared with a rank-128 update.
// Tile-level look-ahead.  The factorisation is a chain of latency-bound launches (one CTA on the diagonal block, ~80 us, then a few GEMM
// tiles), while the trailing updates are the only part with enough tiles to fill the machine.  diag(J+1) needs only block row J+1: the
// panel tile L[J+1,J] = Kw[J+1,J] inv(L_JJ)^T and the update of Kw[J+1,J+1], not the full-height GEMMs of block column J; nor does the
// next super-panel wait for all four of its block columns to receive the K = 512 update.  So:
//   main stream (highest priority): diag(J), row J+1 of the panel, update of the (J+1,J+1) tile (K = 512 from the whole previous
//                                   super-panel when J+1 opens a new one), diag(J+1), ...  -- the row products as chain_gemm32_kernel tiles
//   side stream (middle priority):  rows >= J+2 of panel(J) and of the in-super-panel update, then -- at the end of a super-panel -- the
//                                   K = 512 update of the next super-panel's block columns
//   trail stream (lowest priority): the K = 512 update of all later columns
// The side-stream and trailing GEMMs use 4-stage tiles: 29 against 24 TFLOP/s for 2-stage ones.
// Every output tile is produced by the same k loop as in a one-stream schedule, so the factor is bit-identical to it.
static int32_t blocked_cholesky(agp_ctx* c, double* Kw, double* L, double* Lt, double* Ut, int nb, int64_t ld, int* info, int nvalid) {
  OK((ensure_smem<potrf_trinv128_kernel>(c, PT_SMEM_BYTES)));
  if (nb == 1) {
    potrf_trinv128_kernel<<<1, 256, PT_SMEM_BYTES, c->stream>>>(Kw, L, Lt, Ut, ld, 0, info, std::min(BM, nvalid));
    LAUNCHED(c);
    KCHECK();
    return AGP_OK;
  }
  constexpr int OB = 4;  // inner blocks per super-panel
  cudaStream_t sm = c->stream, ss = c->stream3, st = c->stream2;
  cudaStream_t caller = c->stream;
  const bool part = nb >= 32 && chol_partition(c);  // n >= 4096: below that the factorisation is a millisecond and the split is not worth a second set of streams
  if (part) {  // the chain and the GEMMs move to the two SM partitions; the caller's stream waits for them at the end
    sm = c->pstream_chain;
    ss = c->pstream_side;
    st = c->pstream_trail;
    CU(cudaEventRecord(c->ev_enter, caller));
    CU(cudaStreamWaitEvent(sm, c->ev_enter, 0));
    CU(cudaStreamWaitEvent(ss, c->ev_enter, 0));
    CU(cudaStreamWaitEvent(st, c->ev_enter, 0));
  }
  StreamSwap chain_scope(c, sm);  // launch helpers use c->stream
  auto at = [&](int r, int col) { return (int64_t)col * BM * ld + (int64_t)r * BM; };  // offset of block (r, col)
  bool trail_pending = false, prio_pending = false;
  // development aid (AGP_CHOL_TRACE=1): device timestamps around every diagonal-block kernel of one large factorisation
  static int trace_left = getenv("AGP_CHOL_TRACE") ? 3 : 0;  // the third large factorisation of the process (warm) is traced
  if (trace_left > 0 && nb >= 32) trace_left--;
  const bool trace = getenv("AGP_CHOL_TRACE") && trace_left == 0 && nb >= 32;
  std::vector<cudaEvent_t> marks;
  auto mark = [&]() {
    if (!trace) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, sm);
    marks.push_back(e);
  };
  for (int J0 = 0; J0 < nb; J0 += OB) {
    const int J1 = std::min(nb, J0 + OB), J2 = std::min(nb, J1 + OB);
    for (int J = J0; J < J1; J++) {
      mark();
      potrf_trinv128_kernel<<<1, 256, PT_SMEM_BYTES, sm>>>(Kw + at(J, J), L + at(J, J), Lt + at(J, J), Ut + at(J, J), ld, J * BM, info,
                                                           std::max(0, std::min(BM, nvalid - J * BM)));
      mark();
      LAUNCHED(c);
      KCHECK();
      if (J == nb - 1) break;
      CU(cudaEventRecord(c->ev_diag, sm));
      const int below = nb - 1 - J;  // block rows J+1 .. nb-1
      // ---- main stream: block row J+1 ----
      if (J > J0) CU(cudaStreamWaitEvent(sm, c->ev_side, 0));  // side(J-1): Kw[J+1, J] and Kw[J+1, J+1] carry update(J-1)
      else if (prio_pending) CU(cudaStreamWaitEvent(sm, c->ev_prio, 0));  // K = 512 update of this super-panel's block columns
      chain_gemm32_kernel<<<dim3(4, 4), 128, 0, sm>>>(Kw + at(J + 1, J), ld, Lt + at(J, J), ld, BM, 1, 0, L + at(J + 1, J), ld, 1.0, 0.0);
      LAUNCHED(c);
      KCHECK();
      CU(cudaEventRecord(c->ev_prow, sm));
      if (J + 1 < J1) {
        chain_gemm32_kernel<<<dim3(4, 4), 128, 0, sm>>>(L + at(J + 1, J), ld, L + at(J + 1, J), ld, BM, 0, 1, Kw + at(J + 1, J + 1), ld, -1.0, 1.0);
        LAUNCHED(c);
        KCHECK();
      }
      // ---- side stream: rows >= J+2 of panel(J) and of the update of the remaining block columns (J, J1) ----
      {
        StreamSwap sw(c, ss);
        CU(cudaStreamWaitEvent(ss, c->ev_diag, 0));
        if (below > 1) {
          OK((run_gemm<A_KM, B_KN>(c, below - 1, 2, Kw + at(J + 2, J), ld, Lt + at(J, J), ld, BM, KR_FULL, TS_ALL, epi_store(L + at(J + 2, J), ld, false))));
          const int wcols = J1 - 1 - J;
          if (wcols > 0) {
            CU(cudaStreamWaitEvent(ss, c->ev_prow, 0));  // L[J+1, J] is an operand of column J+1's tiles
            OK((run_gemm<A_KM, B_KN>(c, below - 1, 2 * wcols, L + at(J + 2, J), ld, L + at(J + 1, J), ld, BM, KR_FULL, TS_NBLK_LE1,
                                     epi_store(Kw + at(J + 2, J + 1), ld, false, -1.0, 1.0))));
          }
        }
        CU(cudaEventRecord(c->ev_side, ss));
      }
    }
    prio_pending = false;
    const int rem = nb - J1;
    if (rem <= 0) break;
    const int K = (J1 - J0) * BM;
    // ---- main stream: the diagonal block that opens the next super-panel.  L[J1, J0..J1-2] came from the side stream (the main stream
    // has waited for side(J1-2) above), L[J1, J1-1] from the main stream itself.
    if (trail_pending) CU(cudaStreamWaitEvent(sm, c->ev_trail, 0));
    chain_gemm32_kernel<<<dim3(4, 4), 128, 0, sm>>>(L + at(J1, J0), ld, L + at(J1, J0), ld, K, 0, 1, Kw + at(J1, J1), ld, -1.0, 1.0);
    LAUNCHED(c);
    KCHECK();
    // ---- trail stream: columns >= J2 (needs every row >= J2 of block columns [J0, J1): the side stream up to side(J1-1)) ----
    const int rem2 = nb - J2;
    // ---- side stream: block columns [J1, J2) ----
    {
      StreamSwap sw(c, ss);
      CU(cudaStreamWaitEvent(ss, c->ev_prow, 0));  // L[J1, J1-1]
      if (trail_pending) CU(cudaStreamWaitEvent(ss, c->ev_trail, 0));  // these columns were last written by the previous trailing update
      const int prio_cols = J2 - J1;
      // rows >= J1+1 of the block columns [J1, J2) in one launch (a single wave of tiles once few rows are left: the per-column launches
      // tried first kept the side stream busy for four tile durations and the chain waited for side(J1) behind them)
      if (rem > 1) {
        OK((run_gemm<A_KM, B_KN>(c, rem - 1, 2 * prio_cols, L + at(J1 + 1, J0), ld, L + at(J1, J0), ld, K, KR_FULL, TS_NBLK_LE1, epi_store(Kw + at(J1 + 1, J1), ld, false, -1.0, 1.0))));
      }
      CU(cudaEventRecord(c->ev_prio, ss));
      prio_pending = true;
    }
    if (rem2 > 0) {
      StreamSwap sw(c, st);
      CU(cudaStreamWaitEvent(st, c->ev_side, 0));  // recorded after side(J1-1); the side stream's later work is not waited for
      OK((run_gemm<A_KM, B_KN>(c, rem2, 2 * rem2, L + at(J2, J0), ld, L + at(J2, J0), ld, K, KR_FULL, TS_NBLK_LE, epi_store(Kw + at(J2, J2), ld, false, -1.0, 1.0))));
      CU(cudaEventRecord(c->ev_trail, st));
      trail_pending = true;
    } else {
      trail_pending = false;
    }
  }
  CU(cudaEventRecord(c->ev_side, ss));
  CU(cudaStreamWaitEvent(sm, c->ev_side, 0));
  if (trail_pending) CU(cudaStreamWaitEvent(sm, c->ev_trail, 0));
  if (part) {
    CU(cudaEventRecord(c->ev_leave, sm));
    CU(cudaStreamWaitEvent(caller, c->ev_leave, 0));
  }
  if (trace) {
    mark();
    trace_left = -1;
    cudaStreamSynchronize(sm);
    for (size_t i = 0; i + 1 < marks.size(); i += 2) {
      float t0 = 0.f, t1 = 0.f, t2 = 0.f;
      cudaEventElapsedTime(&t0, marks[0], marks[i]);
      cudaEventElapsedTime(&t1, marks[i], marks[i + 1]);
      cudaEventElapsedTime(&t2, marks[i + 1], marks[i + 2 < marks.size() ? i + 2 : i + 1]);
      fprintf(stderr, "[chol trace v2] J=%2d diag starts %9.1f us, runs %6.1f us, then %6.1f us until the next diag starts\n", (int)(i / 2), 1e3 * t0, 1e3 * t1, 1e3 * t2);
    }
    for (cudaEvent_t e : marks) cudaEventDestroy(e);
  }
  return AGP_OK;
}

// Lt off-diagonal blocks: Lt[J][L<J] = -inv(L_JJ) L[J][L];  Ut[J][L>J] = -(L[L][J] inv(L_JJ))^T
static int32_t build_block_scaled(agp_ctx* c, const double* L, double* Lt, double* Ut, int nb, int64_t ld) {
  if (nb < 2) return AGP_OK;
  // A(m,k) = Lt diag block (column-major, KM); B(k,n) = L[(J*128+k) + n*ld]  (k contiguous: NK)
  OK((run_gemm<A_KM, B_NK>(c, nb, 2 * nb, Lt, ld, L, ld, nb * BM, KR_DIAG, TS_NBLK_LT, epi_store(Lt, ld, false, -1.0))));
  // A(m,k) = Ut diag block = inv^T (KM); B(k,n) = L[n + (J*128+k)*ld]  (n contiguous: KN)
  OK((run_gemm<A_KM, B_KN>(c, nb, 2 * nb, Ut, ld, L, ld, nb * BM, KR_DIAG, TS_NBLK_GT, epi_store(Ut, ld, false, -1.0))));
  return AGP_OK;
}

// ---------------------------------------------------------------------------------------------------
// small element-wise kernels of the SVGP epilogue
// ---------------------------------------------------------------------------------------------------
// KL(q || p) from (mt, Bt, Lk, Lq), cf. SVA.jl:362-373 (DESIGN.md section 2 for the whitened form):
//   0.5 (|Bt|_F^2 + |mt|^2 - M) + sum log diag Lk [centered] - sum log diag Lq
// Stage 1: per-block partial sums of |Bt|_F^2 (fixed order); stage 2: one block adds the O(M) terms.
__global__ void __launch_bounds__(256) kl_partial_kernel(const double* Bt_cm, int64_t n, double* part) {
  __shared__ double sred[8];
  double tr = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double b = Bt_cm[i];
    tr = fma(b, b, tr);
  }
  const double r = block_sum(tr, sred);
  if (threadIdx.x == 0) part[blockIdx.x] = r;
}
__global__ void __launch_bounds__(256) kl_kernel(const double* mt, const double* part, int nparts, const double* Lk, const double* Lq, int M, int Mp,
                                                 int centered, double* out) {
  __shared__ double sred[8];
  double tr = 0.0, mm = 0.0, ldq = 0.0, ldk = 0.0;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) tr += part[i];
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    mm = fma(mt[j], mt[j], mm);
    ldq += log(Lq[(int64_t)j * Mp + j]);
    if (centered) ldk += log(Lk[(int64_t)j * Mp + j]);
  }
  const double a = block_sum(tr, sred);
  const double b = block_sum(mm, sred);
  const double q = block_sum(ldq, sred);
  const double k = block_sum(ldk, sred);
  if (threadIdx.x == 0) out[0] = 0.5 * (a + b - (double)M) + k - q;
}
// zero the strict upper triangle and everything outside the leading M x M block of a column-major Mp x Mp matrix
__global__ void tril_pad_kernel(double* A, int M, int Mp) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x, cidx = blockIdx.y;
  if (r >= Mp) return;
  if (r < cidx || r >= M || cidx >= M) A[(int64_t)cidx * Mp + r] = 0.0;
}

// dLq (column-major M x M, ld = M) from the row-major Mp x Mp cotangent Xrm (lower part used):
//   NonCentered: X - Lq + diag(1/Lq_jj);   Centered: X + diag(1/Lq_jj)
__global__ void finalize_dLq_kernel(const double* Xrm, const double* Lq_cm, int M, int Mp, int centered, double* out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x, cidx = blockIdx.y;
  if (r >= M) return;
  double v = 0.0;
  if (r >= cidx) {
    v = Xrm[(int64_t)r * Mp + cidx];
    const double l = Lq_cm[(int64_t)cidx * Mp + r];
    if (!centered) v -= l;
    if (r == cidx) v += 1.0 / l;
  }
  out[(int64_t)cidx * M + r] = v;
}

// Lbar (row-major) = -tril(V) [- tril(X2) - diag(1/Lk_jj)]
__global__ void build_Lbar_kernel(const double* V, const double* X2, const double* Lk_cm, int Mp, int M, int centered, double* out) {
  const int cidx = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (cidx >= Mp) return;
  double v = 0.0;
  if (r >= cidx) {
    v = -V[(int64_t)r * Mp + cidx];
    if (centered) {
      v -= X2[(int64_t)r * Mp + cidx];
      if (r == cidx && r < M) v -= 1.0 / Lk_cm[(int64_t)r * Mp + r];
    }
  }
  out[(int64_t)r * Mp + cidx] = v;
}

__global__ void set_diag_kernel(double* A, int n, int64_t ld, double v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) A[(int64_t)i * ld + i] = v;
}
__global__ void axpby_kernel(double a, const double* x, double b, const double* y, double* out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = a * x[i] + (y ? b * y[i] : 0.0);
}
// column 0 of a [Mp][64] row-major block <- v ; other columns zero
__global__ void vec_to_rhs_kernel(const double* v, double shift, int M, int Mp, double* rhs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Mp * 64) return;
  const int r = i / 64, cidx = i % 64;
  rhs[i] = (cidx == 0 && r < M) ? v[r] - shift : 0.0;
}
__global__ void rhs_to_vec_kernel(const double* rhs, int Mp, double* v) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < Mp) v[r] = rhs[(int64_t)r * 64];
}
__global__ void __launch_bounds__(256) vec_sum_kernel(const double* v, int n, double* out) {
  __shared__ double sred[8];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += v[i];
  const double r = block_sum(s, sred);
  if (threadIdx.x == 0) out[0] = r;
}

// ---------------------------------------------------------------------------------------------------
// SVGP: per-step preparation
// ---------------------------------------------------------------------------------------------------
// agp_kernel -> KernelParams (validation shared by every entry point that takes a kernel)
static int32_t fill_kernel_params(const agp_kernel* k, int D, int M, KernelParams& kp) {
  if (!k) return fail(AGP_ERR_INVALID, "kernel is NULL");
  if (k->kind < AGP_KERNEL_SE || k->kind > AGP_KERNEL_PRODUCT) return fail(AGP_ERR_UNSUPPORTED, "unsupported kernel kind %d", k->kind);
  if ((k->n_scale != 1 && k->n_scale != D) || !k->inv_lengthscale) return fail(AGP_ERR_INVALID, "kernel.n_scale must be 1 or D");
  memset(&kp, 0, sizeof kp);
  kp.kind = k->kind;
  kp.D = D;
  kp.M = M;
  kp.ard = k->n_scale != 1;
  kp.variance = k->variance;
  kp.c = k->linear_c;
  kp.f0 = 1.0;
  for (int d = 0; d < D; d++) kp.s[d] = k->inv_lengthscale[k->n_scale == 1 ? 0 : d];
  if (kernel_is_composite(k->kind)) {
    if (k->n_components < 1 || k->n_components > AGP_MAX_COMPONENTS || !k->components)
      return fail(AGP_ERR_INVALID, "a kernel sum / product needs 1..%d components", AGP_MAX_COMPONENTS);
    kp.ncomp = k->n_components;
    kp.f0 = k->kind == AGP_KERNEL_SUM ? 0.0 : 1.0;
    for (int i = 0; i < kp.ncomp; i++) {
      const agp_kernel_component& q = k->components[i];
      if (q.kind < AGP_KERNEL_SE || q.kind > AGP_KERNEL_MATERN52)
        return fail(AGP_ERR_UNSUPPORTED, "component %d: only stationary kernels (SqExponential, Matern32, Matern52) can be summed / multiplied on the device", i);
      kp.ckind[i] = q.kind;
      kp.cv[i] = q.variance;
      kp.ca[i] = q.inv_lengthscale * q.inv_lengthscale;
      kp.f0 = k->kind == AGP_KERNEL_SUM ? kp.f0 + q.variance : kp.f0 * q.variance;
    }
  }
  return AGP_OK;
}

// component gradients out of theta (kgrad_finish_kernel) plus the k(x, x) = variance F(0) term of the marginal variances
// (dkxx_sum = sum_n dE/dvar_n * F(0), the SC_DKXX scalar; 0 where there is no such term)
static void write_component_grads(const KernelParams& kp, const double* h_theta, int D, double dkxx_sum, double* dcv, double* dcs) {
  for (int i = 0; i < kp.ncomp; i++) {
    if (dcv) {
      double extra = 0.0;
      if (kp.f0 != 0.0) extra = (dkxx_sum / kp.f0) * kp.variance * (kp.kind == AGP_KERNEL_SUM ? 1.0 : (kp.cv[i] != 0.0 ? kp.f0 / kp.cv[i] : 0.0));
      dcv[i] = h_theta[2 + D + i] + extra;
    }
    if (dcs) dcs[i] = h_theta[2 + D + MAXC + i];
  }
}

static int32_t resolve_params(const agp_svgp_params* p, SvgpState& st) {
  if (!p) return fail(AGP_ERR_INVALID, "params is NULL");
  if (p->M < 1 || p->D < 1 || !p->Z || !p->m || !p->Lq) return fail(AGP_ERR_INVALID, "params: M, D, Z, m, Lq are required");
  if (p->D > MAXD) return fail(AGP_ERR_UNSUPPORTED, "input dimension %d > %d is not supported on device", p->D, MAXD);
  if (p->lik.kind < AGP_LIK_GAUSSIAN || p->lik.kind > AGP_LIK_BERNOULLI_PROBIT) return fail(AGP_ERR_UNSUPPORTED, "unsupported likelihood kind %d", p->lik.kind);
  if (p->parametrization != AGP_NONCENTERED && p->parametrization != AGP_CENTERED) return fail(AGP_ERR_INVALID, "unknown parametrization");
  st.M = p->M;
  st.D = p->D;
  st.Mp = (int)round_up(p->M, BM);
  st.nb = st.Mp / BM;
  st.n_scale = p->kernel.n_scale;
  st.centered = p->parametrization == AGP_CENTERED;
  st.mean_const = p->mean_const;
  st.jitter = p->jitter;
  OK(fill_kernel_params(&p->kernel, p->D, p->M, st.kp));
  if (p->compute_dtype < AGP_COMPUTE_F64 || p->compute_dtype > AGP_COMPUTE_F64_EMU) return fail(AGP_ERR_INVALID, "unknown compute_dtype %d", p->compute_dtype);
  SweepPlan& pl = st.plan;
  pl = SweepPlan{};
  if (p->compute_dtype != AGP_COMPUTE_F64) pl.pts_tile = 2 * BN;
  if (p->compute_dtype == AGP_COMPUTE_F32 || p->compute_dtype == AGP_COMPUTE_F32_TC_SOLVE) {
    pl.s1 = st.Mp >= I8_MIN_ROWS ? ENG_I8 : ENG_DMMA;
    pl.s2 = pl.s4 = pl.s6 = ENG_TF32;
    pl.s5 = p->compute_dtype == AGP_COMPUTE_F32_TC_SOLVE ? ENG_TF32 : ENG_I8;
  } else if (p->compute_dtype == AGP_COMPUTE_F64_EMU && st.Mp >= I8_MIN_ROWS) {
    pl.s2 = pl.s6 = ENG_I8;
  }
  pl.s7_streamed = st.kp.kind >= AGP_KERNEL_SE && st.kp.kind <= AGP_KERNEL_MATERN52;
  st.lp.kind = p->lik.kind;
  st.lp.sigma2 = p->lik.sigma2;
  int method = p->expect.method;
  if (method == AGP_EXPECT_DEFAULT) {
    // GPLikelihoods.DefaultExpectationMethod: analytic for Gaussian and Poisson-exp, else Gauss-Hermite(20)
    method = (p->lik.kind != AGP_LIK_BERNOULLI_LOGIT && p->lik.kind != AGP_LIK_BERNOULLI_PROBIT) ? AGP_EXPECT_ANALYTIC : AGP_EXPECT_GAUSS_HERMITE;
  }
  if (method == AGP_EXPECT_ANALYTIC && (p->lik.kind == AGP_LIK_BERNOULLI_LOGIT || p->lik.kind == AGP_LIK_BERNOULLI_PROBIT))
    return fail(AGP_ERR_UNSUPPORTED, "no analytic expectation for the Bernoulli likelihood");
  st.lp.method = method;
  st.lp.ngh = 0;
  st.lp.seed = 0;
  st.lp.gh = nullptr;
  if (method == AGP_EXPECT_GAUSS_HERMITE) {
    if (p->expect.n_points < 1 || p->expect.n_points > AGP_MAX_GH_POINTS || !p->expect.nodes || !p->expect.weights)
      return fail(AGP_ERR_INVALID, "Gauss-Hermite needs 1..%d nodes and weights from the caller", AGP_MAX_GH_POINTS);
    st.lp.ngh = p->expect.n_points;
  } else if (method == AGP_EXPECT_MONTE_CARLO) {
    if (p->expect.n_points < 1) return fail(AGP_ERR_INVALID, "MonteCarloExpectation needs n_samples >= 1");
    st.lp.ngh = p->expect.n_points;
    st.lp.seed = p->expect.seed;
  } else if (method != AGP_EXPECT_ANALYTIC) {
    return fail(AGP_ERR_UNSUPPORTED, "unsupported expectation method %d", method);
  }
  if (p->lik.kind == AGP_LIK_GAUSSIAN && !(p->lik.sigma2 > 0)) return fail(AGP_ERR_INVALID, "GaussianLikelihood needs sigma2 > 0");
  if (p->lik.kind == AGP_LIK_GAMMA_EXP && !(p->lik.sigma2 > 0)) return fail(AGP_ERR_INVALID, "GammaLikelihood needs alpha > 0");
  return AGP_OK;
}

// Float32 mode: hi / lo planes of the once-per-step operands of the tcgen05 stages -- Bt (column-major memory = the [j][l] operand of
// S2, row-major memory = the [i][j] operand of S4) and the explicit inverse Linv = Lk^-1 (a block TRSM on the identity, as the Laplace
// pullback builds B^-1), transposed to the [j][i] operand of S5.
static int32_t prepare_f32_operands(agp_ctx* c) {
  const int Mp = c->st.Mp;
  const int64_t MM = (int64_t)Mp * Mp;
  if (!t5::encode_tiled_fn()) return fail(AGP_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver (Float32 mode needs TMA tensor maps)");
  DevBuf* planes[] = {&c->fBtc, &c->fBtr, &c->fLi};
  for (DevBuf* b : planes) OK(b->ensure(MM));
  OK(c->W1.ensure(MM));
  OK(c->W2.ensure(MM));
  auto split = [&](const double* in, DevBuf& out) -> int32_t {
    float* hi = reinterpret_cast<float*>(out.p);
    t5::split_planes_kernel<<<1024, 256, 0, c->stream>>>(in, hi, hi + MM, MM);
    LAUNCHED(c);
    KCHECK();
    return AGP_OK;
  };
  OK(split(c->Bt_cm.p, c->fBtc));
  OK(split(c->Bt_rm.p, c->fBtr));
  // W1 (row-major) = I, W1 <- Lk^-1 W1, W2 = W1^T
  OK(fill(c, c->W1.p, MM, 0.0));
  set_diag_kernel<<<(Mp + 255) / 256, 256, 0, c->stream>>>(c->W1.p, Mp, Mp, 1.0);
  LAUNCHED(c);
  KCHECK();
  OK(solve_lk<TR_RHS_FWD>(c, c->W1.p, Mp, Mp / BN));
  // Linv itself (rows l, k = l' contiguous) as seven slice planes: the B operand of the INT8 forward solve (f32sweep.cuh EpiE1)
  OK(c->qLi7.ensure((i8e::S * MM + 7) / 8));
  OK(c->sLi7.ensure(Mp));
  i8e::slice_rows_kernel<i8e::S><<<(Mp + 7) / 8, 256, 0, c->stream>>>(c->W1.p, Mp, Mp, Mp, reinterpret_cast<signed char*>(c->qLi7.p), Mp, MM, c->sLi7.p);
  LAUNCHED(c);
  KCHECK();
  OK(transpose(c, c->W1.p, c->W2.p, Mp, Mp));
  OK(split(c->W2.p, c->fLi));
  // ... and as four INT8 slice planes per row j with a power-of-two row scale: the B operand of the INT8 S5 (f32sweep.cuh EpiE5)
  OK(c->qLi.ensure((i8e::S5_NS * MM + 7) / 8));
  OK(c->sLi.ensure(Mp));
  i8e::slice_rows_kernel<i8e::S5_NS><<<(Mp + 7) / 8, 256, 0, c->stream>>>(c->W2.p, Mp, Mp, Mp, reinterpret_cast<signed char*>(c->qLi.p), Mp, MM, c->sLi.p);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}
// Uploads the parameters and builds every once-per-step operand: zs, zn, Kuu, Lk, Lt, Ut, mt, Bt.
static int32_t prepare_step(agp_ctx* c, const agp_svgp_params* p) {
  SvgpState& st = c->st;
  st.valid = false;
  st.sweep_pending = false;
  OK(resolve_params(p, st));
  CU(cudaSetDevice(c->device));
  const int M = st.M, Mp = st.Mp, D = st.D, nb = st.nb;
  const int64_t MM = (int64_t)Mp * Mp;
  OK(c->z.ensure((int64_t)Mp * D));
  OK(c->zs.ensure((int64_t)Mp * D));
  OK(c->zn.ensure(Mp));
  OK(c->zsp.ensure((int64_t)Mp * (kuf_dp(D) + 2)));
  OK(c->mvec.ensure(Mp));
  OK(c->mt.ensure(Mp));
  OK(c->vec64.ensure((int64_t)Mp * 64));
  OK(c->vec64b.ensure((int64_t)Mp * 64));
  DevBuf* mats[] = {&c->Lq, &c->Kw, &c->Lk, &c->Lt, &c->Ut, &c->Bt_cm, &c->Bt_rm};
  for (DevBuf* b : mats) OK(b->ensure(MM));
  OK(c->small.ensure(64 + 2 * MAXD));
  // host staging: padded m and Lq (lower triangle only)
  st.h_m.assign(Mp, 0.0);
  for (int i = 0; i < M; i++) st.h_m[i] = p->m[i];
  const int ldq = p->ldLq > 0 ? p->ldLq : M;
  for (int j = 0; j < M; j++)
    if (!(p->Lq[(int64_t)j * ldq + j] > 0.0))
      return fail(AGP_ERR_DOMAIN, "q.Sigma Cholesky factor has a non-positive diagonal entry at %d (logdet would throw)", j + 1);
  CU(cudaMemsetAsync(c->z.p, 0, sizeof(double) * Mp * D, c->stream));
  CU(cudaMemcpyAsync(c->z.p, p->Z, sizeof(double) * M * D, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->mvec.p, st.h_m.data(), sizeof(double) * Mp, cudaMemcpyHostToDevice, c->stream));
  // (Lq is uploaded further down, on its own stream, behind the factorisation of Kuu)
  if (st.lp.method == AGP_EXPECT_GAUSS_HERMITE && st.lp.ngh > 0) {
    OK(c->ghbuf.ensure(2 * AGP_MAX_GH_POINTS));
    CU(cudaMemcpyAsync(c->ghbuf.p, p->expect.nodes, sizeof(double) * st.lp.ngh, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->ghbuf.p + AGP_MAX_GH_POINTS, p->expect.weights, sizeof(double) * st.lp.ngh, cudaMemcpyHostToDevice, c->stream));
    st.lp.gh = c->ghbuf.p;
  }
  CU(cudaMemsetAsync(c->d_flags, 0, 4 * sizeof(int), c->stream));
  prep_z_kernel<<<(Mp + 127) / 128, 128, 0, c->stream>>>(c->z.p, c->zs.p, c->zn.p, c->zsp.p, Mp, st.kp);
  LAUNCHED(c);
  KCHECK();
  build_kuu_kernel<<<dim3((Mp + 127) / 128, Mp), 128, 0, c->stream>>>(c->Kw.p, Mp, c->zs.p, c->zn.p, st.jitter, st.kp);
  LAUNCHED(c);
  KCHECK();
  OK(fill(c, c->Lk.p, MM, 0.0));
  OK(fill(c, c->Lt.p, MM, 0.0));
  OK(fill(c, c->Ut.p, MM, 0.0));
  OK(blocked_cholesky(c, c->Kw.p, c->Lk.p, c->Lt.p, c->Ut.p, nb, Mp, c->d_flags, M));
  OK(build_block_scaled(c, c->Lk.p, c->Lt.p, c->Ut.p, nb, Mp));
  // (the Cholesky status word is read together with the results: check_step_flags)
  // Lq: straight from the caller's matrix into the leading M x M block (no host staging of M^2 doubles), then the strict upper triangle
  // and the padding are zeroed on the device (LowerTriangular(A) view, utils.jl:18).  8 MB at M = 1024 from pageable host memory is
  // ~0.8 ms: issued on its own stream AFTER the Kuu kernels have been queued, so that the copy runs under the factorisation (the
  // replicated per-step work is what limits the 8-GPU efficiency of C4).
  CU(cudaMemcpy2DAsync(c->Lq.p, sizeof(double) * Mp, p->Lq, sizeof(double) * ldq, sizeof(double) * M, M, cudaMemcpyHostToDevice, c->stream_copy));
  tril_pad_kernel<<<dim3((Mp + 127) / 128, Mp), 128, 0, c->stream_copy>>>(c->Lq.p, M, Mp);
  LAUNCHED(c);
  KCHECK();
  CU(cudaEventRecord(c->ev_copy, c->stream_copy));
  CU(cudaStreamWaitEvent(c->stream, c->ev_copy, 0));
  if (!st.centered) {
    CU(cudaMemcpyAsync(c->mt.p, c->mvec.p, sizeof(double) * Mp, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaMemcpyAsync(c->Bt_cm.p, c->Lq.p, sizeof(double) * MM, cudaMemcpyDeviceToDevice, c->stream));
    OK(transpose(c, c->Bt_cm.p, c->Bt_rm.p, Mp, Mp));
  } else {
    // mt = Lk^-1 (m - mean(fz));  Bt = Lk^-1 Lq   (SVA.jl:132-133 rewritten in whitened variables)
    vec_to_rhs_kernel<<<(Mp * 64 + 255) / 256, 256, 0, c->stream>>>(c->mvec.p, st.mean_const, M, Mp, c->vec64.p);
    LAUNCHED(c);
    KCHECK();
    OK(solve_lk<TR_RHS_FWD>(c, c->vec64.p, 64, 1));
    rhs_to_vec_kernel<<<(Mp + 255) / 256, 256, 0, c->stream>>>(c->vec64.p, Mp, c->mt.p);
    LAUNCHED(c);
    KCHECK();
    OK(transpose(c, c->Lq.p, c->Bt_rm.p, Mp, Mp));  // row-major Lq as the right-hand side
    OK(solve_lk<TR_RHS_FWD>(c, c->Bt_rm.p, Mp, Mp / BN));
    OK(transpose(c, c->Bt_rm.p, c->Bt_cm.p, Mp, Mp));
  }
  if (st.plan.s2 == ENG_TF32) OK(prepare_f32_operands(c));  // Float32 mode
  st.valid = true;
  return AGP_OK;
}

static int32_t run_kl(agp_ctx* c, double* out) {
  const SvgpState& st = c->st;
  const int nparts = 128;
  double* part = c->vec64.p;  // [Mp*64] right-hand-side scratch, free at this point
  kl_partial_kernel<<<nparts, 256, 0, c->stream>>>(c->Bt_cm.p, (int64_t)st.Mp * st.Mp, part);
  LAUNCHED(c);
  KCHECK();
  kl_kernel<<<1, 256, 0, c->stream>>>(c->mt.p, part, nparts, c->Lk.p, c->Lq.p, st.M, st.Mp, st.centered ? 1 : 0, out);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}

// The status words of a step (Cholesky info, domain flag) are read once, together with the results, instead of
// stalling the stream right after the factorisation.  Synchronises the stream.
static int32_t check_step_flags(agp_ctx* c, bool domain) {
  int h_flags[4];
  CU(cudaMemcpyAsync(h_flags, c->d_flags, sizeof h_flags, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  if (h_flags[0] != 0) return fail_not_pd("cov(fz)", h_flags[0]);
  if (domain && h_flags[1] != 0) return fail(AGP_ERR_DOMAIN, "DomainError: a marginal variance is not positive");
  return AGP_OK;
}

// ---------------------------------------------------------------------------------------------------
// SVGP: the data sweep
// ---------------------------------------------------------------------------------------------------
// slot of the scalar segment (between NSC and the start of g) in which a rank that failed before the collective reports itself
constexpr int SC_PEER_FAILED = NSC + 1;
// layout of the packed reduce buffer
struct RedLayout {
  int64_t scal, g, G, dZ, theta, total;
  RedLayout(int Mp, int D) {
    // every segment starts on a 128-byte boundary (G is a cp.async.16 GEMM operand)
    scal = 0;
    g = round_up(NSC, 16);
    G = g + Mp;
    dZ = G + (int64_t)Mp * Mp;
    theta = round_up(dZ + (int64_t)Mp * D, 16);
    total = theta + theta_size(D);
  }
};

// Points per launch group.  Larger chunks amortise launch gaps and wave tails (measured at C4: 2 waves 1988 ms/step,
// 4 waves 1961, 8 waves 1948); the four M x chunk scratch matrices are capped at ~8 GB.
static int64_t pick_chunk_cols(agp_ctx* c, int64_t count) {
  const int64_t wave = (int64_t)c->sms * 2 * BN;  // one full wave of column tiles at 2 CTAs / SM
  const int64_t by_mem = (int64_t)12e9 / (6 * 8 * std::max(c->st.Mp, BM)) / wave;  // six M x chunk scratch matrices
  int64_t cap = std::min<int64_t>(8, std::max<int64_t>(2, by_mem)) * wave;
  if (const char* e = getenv("AGP_CHUNK_COLS")) cap = std::max<int64_t>(BN, round_up(atoll(e), BN));
  return std::min<int64_t>(cap, round_up(std::max<int64_t>(count, 1), 2 * BN));  // multiples of 128: the tcgen05 stages tile the points by 128
}

static int32_t ensure_sweep_workspace(agp_ctx* c, int64_t cols, bool grad) {
  const SvgpState& st = c->st;
  const SweepPlan& pl = st.plan;
  const int Mp = st.Mp, D = st.D, nb = st.nb;
  const int64_t MM = (int64_t)Mp * Mp;
  if (cols > c->chunk_cols) c->chunk_cols = cols;
  const int64_t cc = c->chunk_cols;
  OK(c->A.ensure((int64_t)Mp * cc));
  OK(c->C.ensure((int64_t)Mp * cc));
  OK(c->saa.ensure(cc));
  OK(c->sam.ensure(cc));
  OK(c->scc_part.ensure((int64_t)(pl.s2 == ENG_I8 ? 4 : 2) * nb * cc));  // column-sum partials of S2 (sweep_s3)
  OK(c->dmu.ensure(cc));
  OK(c->dv.ensure(cc));
  OK(c->sc_part.ensure((cc / 256 + 2) * NSC));
  OK(c->red.ensure(RedLayout(Mp, D).total));
  if (pl.s2 == ENG_TF32) {
    OK(c->fA.ensure((int64_t)Mp * cc));
    OK(c->fC.ensure((int64_t)Mp * cc));
  }
  if (grad && pl.s4 == ENG_TF32) {
    OK(c->fAb.ensure((int64_t)Mp * cc));
    OK(c->fAs.ensure((int64_t)Mp * cc));
  }
  if (grad && pl.s5 == ENG_I8) {
    OK(c->qAb.ensure(((int64_t)i8e::S5_NS * Mp * cc + 7) / 8));
    OK(c->sAb.ensure(2 * cc));  // scales | column maxima
  }
  if (pl.s1 == ENG_I8 || (grad && pl.s7_streamed)) {  // S1 keeps Kuf (and kappa' for the Matern kinds): the INT8 S1 solves from it, S7 reads it
    OK(c->Kf.ensure((int64_t)Mp * cc));
    if (st.kp.kind != AGP_KERNEL_SE) OK(c->DKb.ensure((int64_t)Mp * cc));
  }
  if (pl.s1 == ENG_I8) {
    OK(c->qK.ensure(((int64_t)i8e::S * Mp * cc + 7) / 8));
    OK(c->sK.ensure(cc));
    OK(c->sxx_part.ensure((int64_t)2 * (Mp / 32) * cc));  // saa partials | sam partials, one per 32 inducing rows
  }
  if (grad) {
    OK(c->Ab.ensure((int64_t)Mp * cc));
    OK(c->As.ensure((int64_t)Mp * cc));
    OK(c->gpart.ensure((cc / BN) * Mp));
    const int ntiles = nb * (nb + 1);
    // K-splits of the SYRK: about eight waves of CTAs so that the cheap diagonal tiles (3/8 and 7/8 of a full tile's MMAs)
    // are balanced by the block scheduler (measured at C4: 4 splits / one wave 113 ms per 3e6 points, 32 splits 105 ms);
    // the per-split partial G slices are capped at 512 MB.
    const int by_waves = (8 * 2 * c->sms + ntiles - 1) / ntiles;
    const int by_mem = (int)std::max<int64_t>(1, ((int64_t)512 << 20) / (MM * 8));
    c->nsplit = std::max(1, std::min(std::min(by_waves, by_mem), 32));
    if (pl.s6 == ENG_I8) c->nsplit = std::max<int>(c->nsplit, (int)((round_up(cc, 128) + 16383) / 16384));  // one slab of G per 16384 points
    OK(c->Gpart.ensure((int64_t)c->nsplit * MM));
    c->nslab = (int)std::max<int64_t>((cc + 2047) / 2048, (Mp + 2047) / 2048);
    OK(c->kpart.ensure((int64_t)c->nslab * Mp * kgrad_stride(D)));
    DevBuf* w[] = {&c->W1, &c->W2, &c->W3, &c->W4};
    for (DevBuf* b : w) OK(b->ensure(MM));
  }
  return AGP_OK;
}

static int32_t run_kgrad(agp_ctx* c, const double* Kb, int64_t ld, const double* pts, int npts, int nslab, const double* Kf = nullptr,
                         const double* DK = nullptr) {
  const SvgpState& st = c->st;
  KgradArgs a{};
  a.Kb = Kb;
  a.Kf = Kf;
  a.DK = DK;
  a.ld = ld;
  a.pts = pts;
  a.npts = npts;
  a.zs = c->zs.p;
  a.zn = c->zn.p;
  a.slab = 2048;
  a.part = c->kpart.p;
  a.stride = kgrad_stride(st.D);
  a.Mp = st.Mp;
  a.kp = st.kp;
  const dim3 grid((st.M + 7) / 8, nslab);
  if (Kf) {  // stationary kinds inside the sweep: stream the stored kernel values (kgrad_stream_kernel)
    const bool se = st.kp.kind == AGP_KERNEL_SE;
#define AGP_KSTREAM(DM)                                                                              \
  {                                                                                                  \
    const int sm = KfTile<DM>::value * (DM + 2) * 8;                                                 \
    if (se) {                                                                                        \
      OK((ensure_smem<kgrad_stream_kernel<DM, true>>(c, sm)));                                       \
      kgrad_stream_kernel<DM, true><<<grid, 256, sm, c->stream>>>(a);                                \
    } else {                                                                                         \
      OK((ensure_smem<kgrad_stream_kernel<DM, false>>(c, sm)));                                      \
      kgrad_stream_kernel<DM, false><<<grid, 256, sm, c->stream>>>(a);                               \
    }                                                                                                \
  }
    if (st.D <= 4) AGP_KSTREAM(4)
    else if (st.D <= 8) AGP_KSTREAM(8)
    else if (st.D <= 16) AGP_KSTREAM(16)
    else AGP_KSTREAM(32)
#undef AGP_KSTREAM
    LAUNCHED(c);
    KCHECK();
    return AGP_OK;
  }
  const int smem = 256 * (kuf_dp(st.D) + 2) * 8;
#define AGP_KGRAD_ONE(DM, KD)                                                                                        \
  {                                                                                                                \
    if (smem > 48 * 1024) OK((ensure_smem<kgrad_kernel<DM, 1, KD>>(c, smem)));                                      \
    kgrad_kernel<DM, 1, KD><<<grid, 256, smem, c->stream>>>(a);                                                   \
  }
#define AGP_KGRAD_LAUNCH(DM)                                          \
  switch (st.kp.kind) {                                               \
    case AGP_KERNEL_SE: AGP_KGRAD_ONE(DM, AGP_KERNEL_SE) break;       \
    case AGP_KERNEL_MATERN32: AGP_KGRAD_ONE(DM, AGP_KERNEL_MATERN32) break; \
    case AGP_KERNEL_MATERN52: AGP_KGRAD_ONE(DM, AGP_KERNEL_MATERN52) break; \
    case AGP_KERNEL_LINEAR: AGP_KGRAD_ONE(DM, AGP_KERNEL_LINEAR) break; \
    default: AGP_KGRAD_ONE(DM, AGP_KERNEL_COMPOSITE) break;           \
  }
  if (st.D <= 4) {
    AGP_KGRAD_LAUNCH(4)
  } else if (st.D <= 8) {
    AGP_KGRAD_LAUNCH(8)
  } else if (st.D <= 16) {
    AGP_KGRAD_LAUNCH(16)
  } else {
    AGP_KGRAD_LAUNCH(32)
  }
#undef AGP_KGRAD_LAUNCH
#undef AGP_KGRAD_ONE
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}

static int32_t finish_kgrad(agp_ctx* c, int nslab, double zfac, double* dZ, double* theta) {
  const SvgpState& st = c->st;
  KgradFinishArgs a{};
  a.part = c->kpart.p;
  a.nslab = nslab;
  a.Mp = st.Mp;
  a.stride = kgrad_stride(st.D);
  a.zs = c->zs.p;
  a.zfac = zfac;
  a.dZ = dZ;
  a.theta = theta;
  a.kp = st.kp;
  kgrad_finish_kernel<<<1, 256, 0, c->stream>>>(a);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}

// One tcgen05 3xTF32 GEMM launch (tf32x3.cuh).  Operand planes: hi at p, lo at p + plane; K-major operand = [rows][inner = k],
// MN-major operand = [k rows][inner = m / n].
template <bool AMN, bool BMN, class Epi>
static int32_t launch_t5(agp_ctx* c, dim3 grid, const float* A, int64_t planeA, uint64_t innerA, uint64_t outerA, const float* B, int64_t planeB,
                         uint64_t innerB, uint64_t outerB, const t5::Args& g, const Epi& epi) {
  CUtensorMap mah, mal, mbh, mbl;
  const bool ok = t5::make_map(&mah, A, innerA, outerA, innerA, AMN ? 32 : 128, AMN) && t5::make_map(&mal, A + planeA, innerA, outerA, innerA, AMN ? 32 : 128, AMN) &&
                  t5::make_map(&mbh, B, innerB, outerB, innerB, BMN ? 32 : 128, BMN) && t5::make_map(&mbl, B + planeB, innerB, outerB, innerB, BMN ? 32 : 128, BMN);
  if (!ok) return fail(AGP_ERR_CUDA, "cuTensorMapEncodeTiled failed");
  OK((ensure_smem<t5::tf32x3_gemm_kernel<AMN, BMN, Epi>>(c, t5::SMEM_BYTES)));
  t5::tf32x3_gemm_kernel<AMN, BMN, Epi><<<grid, t5::T5_THREADS, t5::SMEM_BYTES, c->stream>>>(mah, mal, mbh, mbl, g, epi);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}

// One FP64-accurate INT8-slice product (i8emu.cuh).  Each operand is NS slice planes (plane bytes apart) of [rows][k] int8, k contiguous;
// A is tiled by EM rows, B by N rows.
template <class Epi, int NS = i8e::S, int N = i8e::EN>
static int32_t launch_i8(agp_ctx* c, const DevBuf& A, uint64_t rowsA, int64_t planeA, const DevBuf& B, uint64_t rowsB, int64_t planeB, uint64_t k,
                         dim3 grid, const i8e::Args& g, const Epi& epi) {
  CUtensorMap ma, mb;
  if (!i8e::make_map3(&ma, reinterpret_cast<const signed char*>(A.p), k, rowsA, k, planeA, i8e::EM, NS) ||
      !i8e::make_map3(&mb, reinterpret_cast<const signed char*>(B.p), k, rowsB, k, planeB, N, NS))
    return fail(AGP_ERR_CUDA, "cuTensorMapEncodeTiled failed");
  constexpr int smem = i8e::Cfg<NS, N>::smem_bytes;
  OK((ensure_smem<i8e::i8emu_gemm_kernel<Epi, NS, N>>(c, smem)));
  i8e::i8emu_gemm_kernel<Epi, NS, N><<<grid, i8e::E_THREADS, smem, c->stream>>>(ma, mb, g, epi);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}

// S1's arguments for the points [pts, pts + npts): A = Lk^-1 Kuf into X (row stride ldx), column sums into saa / sam
static TrsmArgs s1_args(agp_ctx* c, double* X, int64_t ldx, const double* pts, int npts) {
  TrsmArgs t1{};
  t1.T = c->Lt.p;
  t1.ldt = c->st.Mp;
  t1.nb = c->st.nb;
  t1.X = X;
  t1.ldx = ldx;
  t1.pts = pts;
  t1.npts = npts;
  t1.zsp = c->zsp.p;
  t1.mt = c->mt.p;
  t1.saa = c->saa.p;
  t1.sam = c->sam.p;
  t1.kp = c->st.kp;
  return t1;
}

// The stages of one launch group of the sweep: npts points at pts, padded to ncols columns of the [Mp][chunk_cols] scratch matrices;
// pl is the step's plan at that width (SweepPlan::at_width).

// S1: A = Lk^-1 Kuf with the column sums a^T a and a^T mt.  keep: S7 streams Kuf (and kappa') back from S1.
static int32_t sweep_s1(agp_ctx* c, const SweepPlan& pl, const double* pts, int npts, int ncols, bool keep) {
  const int Mp = c->st.Mp;
  const int64_t ldc = c->chunk_cols, plane = (int64_t)Mp * ldc;
  ProfScope ps(c, PC_TRSM_FWD);
  switch (pl.s1) {
    case ENG_I8: {
      // A = Linv Kuf as an INT8-slice product (7 slices): generator -> Kf (FP64, also S7's input), point-major slices with exact
      // per-point scales, 28 exact slice products, column sums in the epilogue
      OK(launch_s1(c, s1_args(c, c->A.p, ldc, pts, npts), ncols / BN, true, true));
      i8e::transpose_slice_kernel<i8e::S><<<(ncols + 31) / 32, 256, 0, c->stream>>>(c->Kf.p, ldc, Mp, ncols, reinterpret_cast<signed char*>(c->qK.p), Mp,
                                                                                  plane, c->sK.p);
      LAUNCHED(c);
      KCHECK();
      const int nparts = Mp / 32;
      i8e::EpiE1 e1{c->A.p, ldc, c->sK.p, c->sLi7.p, c->mt.p, c->sxx_part.p, c->sxx_part.p + (int64_t)nparts * ldc, ldc};
      // the TF32 planes of A come straight from this epilogue
      e1.Ah = reinterpret_cast<float*>(c->fA.p);
      e1.Al = e1.Ah + plane;
      e1.ldf = Mp;
      OK((launch_i8<i8e::EpiE1>(c, c->qK, ncols, plane, c->qLi7, Mp, (int64_t)Mp * Mp, Mp, dim3(Mp / i8e::EN, ncols / i8e::EM, 1),
                                i8e::Args{Mp, i8e::KM_UPTO_N, 0, 0}, e1)));
      i8e::colsum_reduce_kernel<<<(ncols + 255) / 256, 256, 0, c->stream>>>(c->sxx_part.p, nparts, ldc, ncols, c->saa.p, c->sam.p);
      LAUNCHED(c);
      KCHECK();
      return AGP_OK;
    }
    default:
      return launch_s1(c, s1_args(c, c->A.p, ldc, pts, npts), ncols / BN, keep);
  }
}

// S2: C = Bt^T A with partial column sums of c^T c
static int32_t sweep_s2(agp_ctx* c, const SweepPlan& pl, int ncols) {
  const int Mp = c->st.Mp;
  const int64_t ldc = c->chunk_cols, plane = (int64_t)Mp * ldc, MM = (int64_t)Mp * Mp;
  switch (pl.s2) {
    case ENG_TF32: {
      // point-major hi / lo planes of A (unless the INT8 S1 wrote them), then C = A Bt on the tcgen05 path (f32sweep.cuh)
      float* fA = reinterpret_cast<float*>(c->fA.p);
      float* fC = reinterpret_cast<float*>(c->fC.p);
      if (pl.s1 != ENG_I8) {
        ProfScope ps(c, PC_F32_AUX);
        t5::transpose_split_kernel<<<dim3(ncols / 32, Mp / 32), 256, 0, c->stream>>>(c->A.p, ldc, Mp, ncols, fA, fA + plane, Mp);
        LAUNCHED(c);
        KCHECK();
      }
      ProfScope ps(c, PC_GEMM_BTA);
      t5::EpiF2 e2{fC, fC + plane, Mp, c->scc_part.p, ldc};
      t5::Args g{Mp, t5::KM_FROM_N, 0, 0, t5::MnDesc()};
      return launch_t5<false, false>(c, dim3(ncols / t5::TM, Mp / t5::TN, 1), fA, plane, Mp, ncols, reinterpret_cast<float*>(c->fBtc.p), MM, Mp, Mp, g, e2);
    }
    case ENG_I8: {
      // C[n][j] = sum_{l >= j} A[n][l] Bt[l][j].  The point-major slice planes of A live in the buffer that S6 refills with its own
      // planes later in this launch group.
      ProfScope ps(c, PC_GEMM_BTA);
      OK(c->q6As.ensure(((int64_t)i8e::S * plane + 7) / 8));
      OK(c->sPm.ensure(ldc));
      i8e::transpose_slice_kernel<i8e::S><<<(ncols + 31) / 32, 256, 0, c->stream>>>(c->A.p, ldc, Mp, ncols, reinterpret_cast<signed char*>(c->q6As.p), Mp,
                                                                                  plane, c->sPm.p);
      LAUNCHED(c);
      KCHECK();
      i8e::EpiE2 e2{c->C.p, ldc, c->sPm.p, c->sBt7.p, c->scc_part.p, ldc};
      return launch_i8<i8e::EpiE2>(c, c->q6As, ncols, plane, c->qBt7, Mp, MM, Mp, dim3(Mp / i8e::EN, ncols / i8e::EM, 1), i8e::Args{Mp, i8e::KM_FROM_N, 0, 0}, e2);
    }
    default: {
      // A operand (m=j, k=l) = Bt[l][j] = Bt_rm[l*Mp + j]; nonzero for l >= j
      EpiS2 e2{c->C.p, ldc, c->scc_part.p, ldc};
      ProfScope ps(c, PC_GEMM_BTA);
      return run_gemm<A_KM, B_KN>(c, c->st.nb, ncols / BN, c->Bt_rm.p, Mp, c->A.p, ldc, Mp, KR_UPPER, TS_ALL, e2);
    }
  }
}

// S3: the per-point stage of the points [lo, lo + npts) of X (and y, mu_out, var_out), then (unless predicting) their scalar sums into scal
static int32_t sweep_s3(agp_ctx* c, const SweepPlan& pl, const double* X, const double* y, int64_t lo, int npts, int ncols, bool predict,
                        double* mu_out, double* var_out, double* scal) {
  const SvgpState& st = c->st;
  PerPointArgs pp{};
  pp.saa = c->saa.p;
  pp.sam = c->sam.p;
  pp.scc_part = c->scc_part.p;
  pp.ldp = c->chunk_cols;
  pp.nb = pl.s2 == ENG_TF32 ? 2 * st.nb : pl.s2 == ENG_I8 ? 4 * st.nb : st.nb;  // the column-sum partials S2 wrote
  pp.pts = X + lo * st.D;
  pp.y = y ? y + lo : nullptr;
  pp.npts = npts;
  pp.ncols = ncols;
  pp.scale = st.scale;
  pp.mean_const = st.mean_const;
  pp.kp = st.kp;
  pp.lp = st.lp;
  pp.dmu = c->dmu.p;
  pp.dv = c->dv.p;
  pp.mu_out = mu_out ? mu_out + lo : nullptr;
  pp.var_out = var_out ? var_out + lo : nullptr;
  pp.sc_part = c->sc_part.p;
  pp.flag = c->d_flags + 1;
  pp.predict_only = predict ? 1 : 0;
  pp.point0 = st.point_base + lo;
  const int pblocks = (ncols + PP_POINTS_PER_BLOCK - 1) / PP_POINTS_PER_BLOCK;
  ProfScope ps(c, PC_PERPOINT);
  perpoint_kernel<<<pblocks, 256, 0, c->stream>>>(pp);
  LAUNCHED(c);
  KCHECK();
  if (predict) return AGP_OK;
  const int nsc_used = st.kp.kind == AGP_KERNEL_LINEAR ? SC_DS + st.D : SC_DS;
  scal_reduce_kernel<<<1, 256, 0, c->stream>>>(c->sc_part.p, pblocks, nsc_used, scal);
  LAUNCHED(c);
  KCHECK();
  return AGP_OK;
}

// S4: Ab = dmu (x) mt + 2 dv (Bt C - A), As = dv A (the DMMA epilogue also accumulates g += A dmu)
static int32_t sweep_s4(agp_ctx* c, const SweepPlan& pl, int ncols) {
  const int Mp = c->st.Mp;
  const int64_t ldc = c->chunk_cols, plane = (int64_t)Mp * ldc, MM = (int64_t)Mp * Mp;
  ProfScope ps(c, PC_GEMM_BC);
  switch (pl.s4) {
    case ENG_TF32: {
      float* fA = reinterpret_cast<float*>(c->fA.p);
      float* fC = reinterpret_cast<float*>(c->fC.p);
      float* fAb = reinterpret_cast<float*>(c->fAb.p);
      float* fAs = reinterpret_cast<float*>(c->fAs.p);
      const float* fBtr = reinterpret_cast<float*>(c->fBtr.p);
      const dim3 grid(ncols / t5::TM, Mp / t5::TN, 1);
      t5::Args g{Mp, t5::KM_UPTO_N, 0, 0, t5::MnDesc()};
      if (pl.s5 == ENG_TF32) {
        t5::EpiF4<true> e4{fA, fA + plane, fAb, fAb + plane, fAs, fAs + plane, Mp, c->dmu.p, c->dv.p, c->mt.p, c->Ab.p, ldc};
        return launch_t5<false, false>(c, grid, fC, plane, Mp, ncols, fBtr, MM, Mp, Mp, g, e4);
      }
      t5::EpiF4<false> e4{fA, fA + plane, fAb, fAb + plane, fAs, fAs + plane, Mp, c->dmu.p, c->dv.p, c->mt.p, c->Ab.p, ldc};
      // the column maxima of Ab ride along: the INT8 S5 slices without a pass of its own for them
      CU(cudaMemsetAsync(c->sAb.p + ldc, 0, sizeof(double) * ncols, c->stream));
      e4.abmax = c->sAb.p + ldc;
      return launch_t5<false, false>(c, grid, fC, plane, Mp, ncols, fBtr, MM, Mp, Mp, g, e4);
    }
    default: {
      // A operand (m=j,k=l) = Bt[j][l], l <= j
      EpiS4 e4{c->A.p, c->Ab.p, c->As.p, ldc, c->dmu.p, c->dv.p, c->mt.p, c->gpart.p, Mp};
      return run_gemm<A_KM, B_KN>(c, c->st.nb, ncols / BN, c->Bt_cm.p, Mp, c->C.p, ldc, Mp, KR_LOWER, TS_ALL, e4);
    }
  }
}

// S5: Kb = Lk^-T Ab, in place
static int32_t sweep_s5(agp_ctx* c, const SweepPlan& pl, int ncols) {
  const int Mp = c->st.Mp;
  const int64_t ldc = c->chunk_cols, plane = (int64_t)Mp * ldc, MM = (int64_t)Mp * Mp;
  ProfScope ps(c, PC_TRSM_BWD);
  switch (pl.s5) {
    case ENG_TF32: {
      t5::EpiF5 e5{c->Ab.p, ldc};
      t5::Args g{Mp, t5::KM_FROM_N, 0, 0, t5::MnDesc()};
      return launch_t5<false, false>(c, dim3(ncols / t5::TM, Mp / t5::TN, 1), reinterpret_cast<float*>(c->fAb.p), plane, Mp, ncols,
                                     reinterpret_cast<float*>(c->fLi.p), MM, Mp, Mp, g, e5);
    }
    case ENG_I8: {
      // an exact-accumulation INT8 product with the explicit inverse: Ab (FP64, inducing-major, from the S4 epilogue) is cut into
      // S5_NS slice planes per point, the product overwrites Ab with Kb
      i8e::transpose_slice_kernel<i8e::S5_NS><<<(ncols + 31) / 32, 256, 0, c->stream>>>(c->Ab.p, ldc, Mp, ncols, reinterpret_cast<signed char*>(c->qAb.p), Mp,
                                                                                      plane, c->sAb.p, c->sAb.p + ldc);
      LAUNCHED(c);
      KCHECK();
      i8e::EpiE5 e5{c->Ab.p, ldc, c->sAb.p, c->sLi.p};
      return launch_i8<i8e::EpiE5, i8e::S5_NS, i8e::S5_N>(c, c->qAb, ncols, plane, c->qLi, Mp, MM, Mp, dim3(Mp / i8e::S5_N, ncols / i8e::EM, 1),
                                                          i8e::Args{Mp, i8e::KM_FROM_N, 0, 0}, e5);
    }
    default:
      return solve_lk<TR_RHS_BWD>(c, c->Ab.p, ldc, ncols / BN);
  }
}

// S6: G += As A^T, one partial G per split of the points.  After a TF32 S4, whose epilogue leaves it out, g += A dmu follows.
static int32_t sweep_s6(agp_ctx* c, const SweepPlan& pl, int ncols) {
  const int Mp = c->st.Mp, nb = c->st.nb;
  const int64_t ldc = c->chunk_cols, plane = (int64_t)Mp * ldc;
  float* fA = reinterpret_cast<float*>(c->fA.p);
  {
    ProfScope ps(c, PC_SYRK);
    switch (pl.s6) {
      case ENG_TF32: {
        const int kchunk = (int)round_up((ncols + c->nsplit - 1) / c->nsplit, t5::TM);
        const int nz = (ncols + kchunk - 1) / kchunk;
        t5::EpiF6 e6{c->Gpart.p, Mp};
        t5::Args g{ncols, t5::KM_SPLIT, kchunk, 1, t5::MnDesc()};
        OK((launch_t5<true, true>(c, dim3(Mp / t5::TM, Mp / t5::TN, nz), reinterpret_cast<float*>(c->fAs.p), plane, Mp, ncols, fA, plane, Mp, ncols, g, e6)));
        break;
      }
      case ENG_I8: {
        // Operands are already K-major (points contiguous): row maxima -> power-of-two scales -> seven 7-bit slice planes each for As
        // (A operand, 128-row tiles) and A (B operand, 64-row tiles); one slab of 16384 points per blockIdx.z (INT32 accumulators:
        // 7 * 127^2 * 16384 < 2^31), partial G per slab, summed in a fixed order with the other slabs
        const int64_t ldk = round_up(ncols, 128), pbytes = (int64_t)Mp * ldk;
        OK(c->q6A.ensure(((int64_t)i8e::S * pbytes + 7) / 8));
        OK(c->q6As.ensure(((int64_t)i8e::S * pbytes + 7) / 8));
        OK(c->s6.ensure(4 * (int64_t)Mp));
        double* sA = c->s6.p;
        double* sAs = c->s6.p + Mp;
        unsigned long long* mx = reinterpret_cast<unsigned long long*>(c->s6.p + 2 * Mp);
        CU(cudaMemsetAsync(mx, 0, sizeof(unsigned long long) * 2 * Mp, c->stream));
        const int seg = 8192;
        const dim3 gmx((ncols + seg - 1) / seg, Mp / 8);
        i8e::rowmax_kernel<<<gmx, 256, 0, c->stream>>>(c->A.p, ldc, Mp, ncols, seg, mx);
        LAUNCHED(c);
        i8e::rowmax_kernel<<<gmx, 256, 0, c->stream>>>(c->As.p, ldc, Mp, ncols, seg, mx + Mp);
        LAUNCHED(c);
        const dim3 gsl((unsigned)((ldk + 1023) / 1024), Mp);
        i8e::slice_rows2d_kernel<i8e::S><<<gsl, 256, 0, c->stream>>>(c->A.p, ldc, ncols, reinterpret_cast<signed char*>(c->q6A.p), ldk, pbytes, mx, sA);
        LAUNCHED(c);
        i8e::slice_rows2d_kernel<i8e::S><<<gsl, 256, 0, c->stream>>>(c->As.p, ldc, ncols, reinterpret_cast<signed char*>(c->q6As.p), ldk, pbytes, mx + Mp, sAs);
        LAUNCHED(c);
        KCHECK();
        const int kchunk = 16384, nz = (int)((ldk + kchunk - 1) / kchunk);
        if (nz > c->nsplit) return fail(AGP_ERR_ALLOC, "S6 (INT8): %d slabs of G needed, %d allocated", nz, c->nsplit);
        i8e::EpiE6 e6{c->Gpart.p, Mp, sAs, sA};
        OK((launch_i8<i8e::EpiE6>(c, c->q6As, Mp, pbytes, c->q6A, Mp, pbytes, ldk, dim3(Mp / i8e::EN, Mp / i8e::EM, nz),
                                  i8e::Args{(int)ldk, i8e::KM_SPLIT, kchunk, 1}, e6)));
        break;
      }
      default: {
        SyrkArgs s{};
        s.As = c->As.p;
        s.A = c->A.p;
        s.ld = ldc;
        s.ncols = ncols;
        s.kchunk = (int)round_up((ncols + c->nsplit - 1) / c->nsplit, BK);
        s.G = c->Gpart.p;
        s.Mp = Mp;
        using Cfg = StageCfg<A_MK, B_NK>;
        OK((ensure_smem<syrk_kernel>(c, Cfg::smem_bytes)));
        syrk_kernel<<<dim3(nb * (nb + 1), c->nsplit), NTHREADS, Cfg::smem_bytes, c->stream>>>(s);
        LAUNCHED(c);
        KCHECK();
      }
    }
  }
  if (pl.s4 == ENG_TF32) {
    ProfScope ps(c, PC_F32_AUX);
    const int slab = 512, nslab = (ncols + slab - 1) / slab;
    t5::gvec_kernel<<<dim3((Mp / 4 + 255) / 256, nslab), 256, 0, c->stream>>>(fA, fA + plane, Mp, Mp, c->dmu.p, ncols, slab, c->gpart.p, Mp);
    LAUNCHED(c);
    KCHECK();
  }
  return AGP_OK;
}

// S7: contraction of Kb with the kernel derivatives
static int32_t sweep_s7(agp_ctx* c, const SweepPlan& pl, const double* pts, int npts) {
  const bool dk = pl.s7_streamed && c->st.kp.kind != AGP_KERNEL_SE;
  ProfScope ps(c, PC_KGRAD);
  return run_kgrad(c, c->Ab.p, c->chunk_cols, pts, npts, (npts + 2047) / 2048, pl.s7_streamed ? c->Kf.p : nullptr, dk ? c->DKb.p : nullptr);
}

// local reductions of the reverse pass's partial sums into the packed reduce buffer
static int32_t sweep_reduce(agp_ctx* c, const RedLayout& rl) {
  const int Mp = c->st.Mp;
  const int64_t MM = (int64_t)Mp * Mp;
  sum_slices_kernel<<<(Mp + 255) / 256, 256, 0, c->stream>>>(c->gpart.p, (int)(c->chunk_cols / BN), Mp, Mp, c->red.p + rl.g);
  LAUNCHED(c);
  KCHECK();
  sum_slices_kernel<<<1024, 256, 0, c->stream>>>(c->Gpart.p, c->nsplit, MM, MM, c->red.p + rl.G);
  LAUNCHED(c);
  KCHECK();
  return finish_kgrad(c, c->nslab, 1.0, c->red.p + rl.dZ, c->red.p + rl.theta);
}

// forward (+ backward) sweep over points [offset, offset+count) of ds.  predict != 0: only S1-S3 writing mu/var.
static int32_t sweep_points(agp_ctx* c, const double* X, const double* y, int64_t count, bool grad, bool predict, double* mu_out,
                            double* var_out) {
  const SweepPlan& pl = c->st.plan;
  const int Mp = c->st.Mp, D = c->st.D;
  const int64_t MM = (int64_t)Mp * Mp;
  const int64_t cols = pick_chunk_cols(c, count);
  OK(ensure_sweep_workspace(c, cols, grad));
  const int64_t ldc = c->chunk_cols;
  RedLayout rl(Mp, D);
  if (!predict) {
    OK(fill(c, c->red.p, rl.total, 0.0));
    if (grad) {
      OK(fill(c, c->gpart.p, (ldc / BN) * Mp, 0.0));
      OK(fill(c, c->Gpart.p, (int64_t)c->nsplit * MM, 0.0));
      OK(fill(c, c->kpart.p, (int64_t)c->nslab * Mp * kgrad_stride(D), 0.0));
    }
  }
  if (pl.s2 == ENG_I8) {  // slices of the rows of Bt^T (columns of Bt, contiguous in the column-major copy), one scale per column
    OK(c->qBt7.ensure(((int64_t)i8e::S * MM + 7) / 8));
    OK(c->sBt7.ensure(Mp));
    i8e::slice_rows_kernel<i8e::S><<<(Mp + 7) / 8, 256, 0, c->stream>>>(c->Bt_cm.p, Mp, Mp, Mp, reinterpret_cast<signed char*>(c->qBt7.p), Mp, MM, c->sBt7.p);
    LAUNCHED(c);
    KCHECK();
  }
  for (int64_t lo = 0; lo < count; lo += cols) {
    const int npts = (int)std::min<int64_t>(cols, count - lo);
    const int ncols = (int)round_up(npts, pl.pts_tile);
    const SweepPlan gp = pl.at_width(ncols);
    OK(sweep_s1(c, gp, X + lo * D, npts, ncols, grad && gp.s7_streamed));
    OK(sweep_s2(c, gp, ncols));
    OK(sweep_s3(c, gp, X, y, lo, npts, ncols, predict, mu_out, var_out, c->red.p + rl.scal));
    if (predict || !grad) continue;
    OK(sweep_s4(c, gp, ncols));
    OK(sweep_s5(c, gp, ncols));
    OK(sweep_s6(c, gp, ncols));
    OK(sweep_s7(c, gp, X + lo * D, npts));
  }
  if (predict || !grad) return AGP_OK;
  return sweep_reduce(c, rl);
}

static int32_t check_dataset(agp_ctx* c, agp_dataset* ds, int64_t offset, int64_t count, int D) {
  if (!c || !ds) return fail(AGP_ERR_INVALID, "NULL context or dataset");
  if (ds->ctx != c) return fail(AGP_ERR_INVALID, "dataset belongs to another context");
  if (ds->D != D) return fail(AGP_ERR_INVALID, "dataset dimension %d != params.D %d", ds->D, D);
  // an empty shard (count == 0) is legal for a rank of a data-parallel job with fewer points than ranks: it contributes zeros
  const int64_t min_count = (c->comm && c->nranks > 1) ? 0 : 1;
  if (offset < 0 || count < min_count || offset + count > ds->N)
    return fail(AGP_ERR_INVALID, "points [%lld, %lld) outside the dataset (N=%lld)", (long long)offset, (long long)(offset + count), (long long)ds->N);
  return AGP_OK;
}

extern "C" int32_t agp_svgp_sweep(agp_ctx* c, agp_dataset* ds, int64_t offset, int64_t count, const agp_svgp_params* p,
                                  double num_data, int64_t global_batch, int32_t want_grad) {
  if (!c || !p) return fail(AGP_ERR_INVALID, "agp_svgp_sweep: NULL argument");
  if (c->comm && c->nranks > 1 && global_batch <= 0)
    return fail(AGP_ERR_INVALID, "with a communicator attached global_batch (the batch size summed over all ranks) is required: "
                                 "num_data / count of one shard would scale the ELBO by the number of ranks");
  OK(check_dataset(c, ds, offset, count, p->D));
  {
    ProfScope ps(c, PC_PREPARE);
    OK(prepare_step(c, p));
  }
  SvgpState& st = c->st;
  const int64_t gb = global_batch > 0 ? global_batch : count;
  st.scale = (num_data > 0 ? num_data : (double)gb) / (double)gb;  // SVA.jl:357-358
  st.want_grad = want_grad;
  st.point_base = offset + ((long long)c->rank << 40);  // distinct Monte-Carlo streams per rank
  OK(sweep_points(c, ds->X + offset * ds->D, ds->y + offset, count, want_grad != 0, false, nullptr, nullptr));
  st.sweep_pending = true;
  return AGP_OK;
}

extern "C" int32_t agp_svgp_reduce_buffer(agp_ctx* c, void** dptr, int64_t* n) {
  if (!c || !c->st.valid || !c->st.sweep_pending) return fail(AGP_ERR_INVALID, "agp_svgp_reduce_buffer: no sweep pending");
  RedLayout rl(c->st.Mp, c->st.D);
  if (dptr) *dptr = c->red.p;
  if (n) *n = c->st.want_grad ? rl.total : rl.g;
  CU(cudaStreamSynchronize(c->stream));  // the caller's collective runs on its own stream
  return AGP_OK;
}

// ---------------------------------------------------------------------------------------------------
// SVGP: replicated epilogue (KL, Cholesky pullback, Kuu part of dZ / dtheta)
// ---------------------------------------------------------------------------------------------------
extern "C" int32_t agp_svgp_finish(agp_ctx* c, double* elbo_out, agp_svgp_grads* go) {
  // (st.valid alone is also set by prior_kl / posterior / mean_and_var, whose prepare_step leaves no reduce buffer behind)
  if (!c || !c->st.valid || !c->st.sweep_pending) return fail(AGP_ERR_INVALID, "agp_svgp_finish: no sweep pending");
  c->st.sweep_pending = false;
  CU(cudaSetDevice(c->device));
  ProfScope ps_finish(c, PC_FINISH);
  SvgpState& st = c->st;
  const int M = st.M, Mp = st.Mp, D = st.D, nb = st.nb;
  const int64_t MM = (int64_t)Mp * Mp;
  RedLayout rl(Mp, D);
  double* red = c->red.p;
  double* small = c->small.p;  // [0] KL, [1] sum(mbar) (centered)
  OK(run_kl(c, small));
  std::vector<double> h_scal(rl.g), h_small(4, 0.0);
  if (!st.want_grad || !go) {
    CU(cudaMemcpyAsync(h_scal.data(), red + rl.scal, sizeof(double) * rl.g, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(h_small.data(), small, sizeof(double) * 1, cudaMemcpyDeviceToHost, c->stream));
    int h_flags[4];
    CU(cudaMemcpyAsync(h_flags, c->d_flags, sizeof h_flags, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (h_scal[SC_PEER_FAILED] != 0.0) return fail(AGP_ERR_NCCL, "%d peer rank(s) failed before the all-reduce; the result is invalid", (int)h_scal[SC_PEER_FAILED]);
    if (h_flags[0] != 0) return fail_not_pd("cov(fz)", h_flags[0]);
    if (h_flags[1] != 0) return fail(AGP_ERR_DOMAIN, "DomainError: a marginal variance is not positive");
    if (elbo_out) *elbo_out = h_scal[SC_E] * st.scale - h_small[0];
    return AGP_OK;
  }
  double* g = red + rl.g;
  double* G = red + rl.G;
  double* dZ = red + rl.dZ;
  double* theta = red + rl.theta;
  double *W1 = c->W1.p, *W2 = c->W2.p, *W3 = c->W3.p, *W4 = c->W4.p;
  // G: lower tiles -> full symmetric
  symmetrize_from_lower_kernel<<<dim3((Mp + 127) / 128, Mp), 128, 0, c->stream>>>(G, Mp, Mp);
  LAUNCHED(c);
  KCHECK();
  // W1 = P1 = Bt Bt^T - I
  OK((run_gemm<A_KM, B_KN>(c, nb, Mp / BN, c->Bt_cm.p, Mp, c->Bt_cm.p, Mp, Mp, KR_FULL, TS_ALL,
                           epi_store(W1, Mp, false, 1.0, 0.0, MASK_NONE, -1.0))));
  // W2 (row-major) = Asum = mt g^T + 2 P1 G
  OK((run_gemm<A_KM, B_KN>(c, nb, Mp / BN, W1, Mp, G, Mp, Mp, KR_FULL, TS_ALL,
                           epi_store(W2, Mp, true, 2.0, 0.0, MASK_NONE, 0.0, c->mt.p, g, 1.0))));
  // W2 <- V = Lk^-T Asum
  OK(solve_lk<TR_RHS_BWD>(c, W2, Mp, Mp / BN));
  // W3 (row-major) = Bt-bar = tril(2 G Bt) [- Bt if centered]
  //   B operand (k, n) = Bt[k][n] = Bt_rm[k*Mp + n]
  OK((run_gemm<A_KM, B_KN>(c, nb, Mp / BN, G, Mp, c->Bt_rm.p, Mp, Mp, KR_FULL, TS_ALL, epi_store(W3, Mp, true, 2.0, 0.0, MASK_LOWER))));
  double* dLq_src = W3;
  if (st.centered) {
    // Bt-bar -= Bt ;  mt-bar = g - mt
    axpby_kernel<<<1024, 256, 0, c->stream>>>(1.0, W3, -1.0, c->Bt_rm.p, W3, MM);
    LAUNCHED(c);
    KCHECK();
    axpby_kernel<<<(Mp + 255) / 256, 256, 0, c->stream>>>(1.0, g, -1.0, c->mt.p, c->vec64b.p, Mp);  // mt-bar in vec64b[0..Mp)
    LAUNCHED(c);
    KCHECK();
    // m-bar = Lk^-T mt-bar
    vec_to_rhs_kernel<<<(Mp * 64 + 255) / 256, 256, 0, c->stream>>>(c->vec64b.p, 0.0, Mp, Mp, c->vec64.p);
    LAUNCHED(c);
    KCHECK();
    OK(solve_lk<TR_RHS_BWD>(c, c->vec64.p, 64, 1));
    rhs_to_vec_kernel<<<(Mp + 255) / 256, 256, 0, c->stream>>>(c->vec64.p, Mp, c->vec64b.p + Mp);  // m-bar in vec64b[Mp..2Mp)
    LAUNCHED(c);
    KCHECK();
    vec_sum_kernel<<<1, 256, 0, c->stream>>>(c->vec64b.p + Mp, M, small + 1);
    LAUNCHED(c);
    KCHECK();
    // W3 <- Y = Lk^-T Bt-bar (row-major, in place)
    OK(solve_lk<TR_RHS_BWD>(c, W3, Mp, Mp / BN));
    // W4 (row-major) = X2 = Y Bt^T + m-bar mt^T ;  A operand (m,k) = Y[m][k] row-major (MK); B (k,n) = Bt[n][k] = Bt_cm[n + k*Mp]
    OK((run_gemm<A_MK, B_KN>(c, nb, Mp / BN, W3, Mp, c->Bt_cm.p, Mp, Mp, KR_FULL, TS_ALL,
                             epi_store(W4, Mp, true, 1.0, 0.0, MASK_NONE, 0.0, c->vec64b.p + Mp, c->mt.p, 1.0))));
  }
  // dLq_src (W3) is final from here on: its read-back (M^2 doubles, the largest output) goes to the copy stream below and runs under the
  // Cholesky pullback and the Kuu part of the kernel gradient
  if (go->dLq) CU(cudaEventRecord(c->ev_copy, c->stream));
  // W1 (row-major) = Lk-bar
  build_Lbar_kernel<<<dim3((Mp + 127) / 128, Mp), 128, 0, c->stream>>>(W2, W4, c->Lk.p, Mp, M, st.centered ? 1 : 0, W1);
  LAUNCHED(c);
  KCHECK();
  // W2 (row-major) = Phi(Lk^T Lk-bar);  A operand (m,k) = Lk[k][m] = Lk_cm[k + m*Mp] (MK), nonzero for k >= m
  OK((run_gemm<A_MK, B_KN>(c, nb, Mp / BN, c->Lk.p, Mp, W1, Mp, Mp, KR_UPPER, TS_ALL, epi_store(W2, Mp, true, 1.0, 0.0, MASK_PHI))));
  // Y1 = Lk^-T W2 ; Y2 = Lk^-T Y1^T ; Kuu-bar = (Y2 + Y2^T)/2
  OK(solve_lk<TR_RHS_BWD>(c, W2, Mp, Mp / BN));
  OK(transpose(c, W2, W1, Mp, Mp));
  OK(solve_lk<TR_RHS_BWD>(c, W1, Mp, Mp / BN));
  OK(transpose(c, W1, W2, Mp, Mp));
  sym_average_kernel<<<1024, 256, 0, c->stream>>>(W1, W2, W4, MM);  // W4 = Kuu-bar (symmetric)
  LAUNCHED(c);
  KCHECK();
  // Kuu part of dZ / dtheta: contraction with k(Z, Z); both arguments move -> zfac = 2
  const int nslab_z = (M + 2047) / 2048;
  OK(fill(c, c->kpart.p, (int64_t)nslab_z * Mp * kgrad_stride(D), 0.0));
  OK(run_kgrad(c, W4, Mp, c->z.p, M, nslab_z));
  OK(finish_kgrad(c, nslab_z, 2.0, dZ, theta));
  // outputs
  std::vector<double> h_theta(theta_size(D)), h_dZ((int64_t)Mp * D), h_vec(2 * (int64_t)Mp), h_g(Mp);
  std::vector<double> h_dLq;
  if (go->dLq) {
    // issued before the small read-backs: a copy into pageable host memory holds the host until it is done, and by now every kernel of
    // the epilogue is queued on the main stream
    OK(c->A.ensure((int64_t)M * M));  // reuse chunk scratch as the staging area
    CU(cudaStreamWaitEvent(c->stream_copy, c->ev_copy, 0));
    finalize_dLq_kernel<<<dim3((M + 127) / 128, M), 128, 0, c->stream_copy>>>(dLq_src, c->Lq.p, M, Mp, st.centered ? 1 : 0, c->A.p);
    LAUNCHED(c);
    KCHECK();
    CU(cudaMemcpyAsync(go->dLq, c->A.p, sizeof(double) * M * M, cudaMemcpyDeviceToHost, c->stream_copy));
  }
  CU(cudaMemcpyAsync(h_scal.data(), red + rl.scal, sizeof(double) * rl.g, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(h_small.data(), small, sizeof(double) * 2, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(h_theta.data(), theta, sizeof(double) * theta_size(D), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(h_dZ.data(), dZ, sizeof(double) * Mp * D, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(h_g.data(), g, sizeof(double) * Mp, cudaMemcpyDeviceToHost, c->stream));
  if (st.centered) CU(cudaMemcpyAsync(h_vec.data(), c->vec64b.p, sizeof(double) * 2 * Mp, cudaMemcpyDeviceToHost, c->stream));
  int h_flags[4];
  CU(cudaMemcpyAsync(h_flags, c->d_flags, sizeof h_flags, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  if (go->dLq) CU(cudaStreamSynchronize(c->stream_copy));
  if (h_scal[SC_PEER_FAILED] != 0.0) return fail(AGP_ERR_NCCL, "%d peer rank(s) failed before the all-reduce; the result is invalid", (int)h_scal[SC_PEER_FAILED]);
  if (h_flags[0] != 0) return fail_not_pd("cov(fz)", h_flags[0]);
  if (h_flags[1] != 0) return fail(AGP_ERR_DOMAIN, "DomainError: a marginal variance is not positive");
  if (elbo_out) *elbo_out = h_scal[SC_E] * st.scale - h_small[0];
  if (go->dm) {
    for (int i = 0; i < M; i++) go->dm[i] = st.centered ? h_vec[Mp + i] : h_g[i] - st.h_m[i];
  }
  if (go->dZ) memcpy(go->dZ, h_dZ.data(), sizeof(double) * M * D);
  if (go->dvariance) *go->dvariance = h_theta[0] + h_scal[SC_DKXX];
  if (go->dlinear_c) *go->dlinear_c = h_theta[1] + h_scal[SC_DC];
  if (go->dinv_lengthscale) {
    const bool linear = st.kp.kind == AGP_KERNEL_LINEAR;
    if (st.n_scale == 1) {
      double s = 0.0;
      for (int d = 0; d < D; d++) s += h_theta[2 + d] + (linear ? h_scal[SC_DS + d] : 0.0);
      go->dinv_lengthscale[0] = s;
    } else {
      for (int d = 0; d < D; d++) go->dinv_lengthscale[d] = h_theta[2 + d] + (linear ? h_scal[SC_DS + d] : 0.0);
    }
  }
  if (kernel_is_composite(st.kp.kind)) write_component_grads(st.kp, h_theta.data(), D, h_scal[SC_DKXX], go->dcomp_variance, go->dcomp_inv_lengthscale);
  if (go->dmean_const) *go->dmean_const = h_scal[SC_DMU] - (st.centered ? h_small[1] : 0.0);
  if (go->dlik_sigma2) *go->dlik_sigma2 = h_scal[SC_DS2];
  return AGP_OK;
}

static int32_t allreduce_if_needed(agp_ctx* c) {
  if (!c->comm || c->nranks == 1) return AGP_OK;
  RedLayout rl(c->st.Mp, c->st.D);
  const size_t n = c->st.want_grad ? (size_t)rl.total : (size_t)rl.g;
  ProfScope ps(c, PC_ALLREDUCE);
  ncclResult_t r = g_nccl.AllReduce(c->red.p, c->red.p, n, ncclDouble, ncclSum, c->comm, c->stream);
  if (r != ncclSuccess) return fail(AGP_ERR_NCCL, "ncclAllReduce: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
  return AGP_OK;
}

// A rank whose sweep failed locally (allocation, CUDA error, a bad shard) must still enter the collective, or its peers block
// in ncclAllReduce forever: it contributes a zero buffer with SC_PEER_FAILED = 1, the peers see the non-zero slot in
// agp_svgp_finish and fail with AGP_ERR_NCCL, and this rank returns its own error.  (Argument errors that every rank detects
// identically -- NULL pointers, global_batch <= 0 -- return before the collective on all of them.)
static void signal_failure_to_peers(agp_ctx* c, const agp_svgp_params* p, bool want_grad) {
  if (!c || !c->comm || c->nranks < 2 || !p || p->M < 1 || p->D < 1 || p->D > MAXD) return;
  const std::string saved = g_err;
  const int Mp = (int)round_up(p->M, BM);
  RedLayout rl(Mp, p->D);
  if (cudaSetDevice(c->device) == cudaSuccess && c->red.ensure(rl.total) == AGP_OK) {
    const double one = 1.0;
    cudaMemsetAsync(c->red.p, 0, sizeof(double) * rl.total, c->stream);
    cudaMemcpyAsync(c->red.p + SC_PEER_FAILED, &one, sizeof one, cudaMemcpyHostToDevice, c->stream);
    g_nccl.AllReduce(c->red.p, c->red.p, want_grad ? (size_t)rl.total : (size_t)rl.g, ncclDouble, ncclSum, c->comm, c->stream);
    cudaStreamSynchronize(c->stream);
  }
  g_err = saved;
}

extern "C" int32_t agp_svgp_elbo_grad(agp_ctx* c, agp_dataset* ds, int64_t offset, int64_t count, const agp_svgp_params* p,
                                      double num_data, int64_t global_batch, double* elbo_out, agp_svgp_grads* go) {
  const int32_t s = agp_svgp_sweep(c, ds, offset, count, p, num_data, global_batch, go ? 1 : 0);
  if (s != AGP_OK) {
    if (c && !(c->comm && c->nranks > 1 && global_batch <= 0)) signal_failure_to_peers(c, p, go != nullptr);
    return s;
  }
  OK(allreduce_if_needed(c));
  return agp_svgp_finish(c, elbo_out, go);
}

// Flat-vector form (SURVEY.md section 8f-3): [variance | inv_lengthscale (n_scale) | linear_c | mean_const | lik parameter |
// Z (M*D, point-major) | m (M) | Lq (M*M, column-major) | kernel sums / products: component variances (n_components) |
// component inverse lengthscales (n_components)] in, the gradient in the same layout out.
static int flat_ncomp(const agp_svgp_params* p) {
  return (kernel_is_composite(p->kernel.kind) && p->kernel.n_components >= 1 && p->kernel.n_components <= AGP_MAX_COMPONENTS && p->kernel.components) ? p->kernel.n_components : 0;
}
static int64_t flat_size(const agp_svgp_params* p) {
  if (!p || p->M < 1 || p->D < 1 || p->kernel.n_scale < 1) return 0;
  return 4 + (int64_t)p->kernel.n_scale + (int64_t)p->M * p->D + p->M + (int64_t)p->M * p->M + 2 * flat_ncomp(p);
}
extern "C" int32_t agp_svgp_flat_size(const agp_svgp_params* p, int64_t* n_out) {
  const int64_t n = flat_size(p);
  if (n == 0 || !n_out) return fail(AGP_ERR_INVALID, "agp_svgp_flat_size: template needs M, D and kernel.n_scale");
  *n_out = n;
  return AGP_OK;
}
extern "C" int32_t agp_svgp_elbo_grad_flat(agp_ctx* c, agp_dataset* ds, int64_t offset, int64_t count, const agp_svgp_params* tmpl,
                                           const double* flat, double num_data, int64_t global_batch, double* elbo_out, double* flat_grad) {
  if (!tmpl || !flat) return fail(AGP_ERR_INVALID, "agp_svgp_elbo_grad_flat: NULL argument");
  if (flat_size(tmpl) == 0) return fail(AGP_ERR_INVALID, "agp_svgp_elbo_grad_flat: template needs M, D and kernel.n_scale");
  agp_svgp_params p = *tmpl;
  const int ns = p.kernel.n_scale, M = p.M, D = p.D;
  const double* f = flat;
  p.kernel.variance = f[0];
  p.kernel.inv_lengthscale = f + 1;
  p.kernel.linear_c = f[1 + ns];
  p.mean_const = f[2 + ns];
  p.lik.sigma2 = f[3 + ns];
  p.Z = f + 4 + ns;
  p.m = p.Z + (int64_t)M * D;
  p.Lq = p.m + M;
  p.ldLq = M;
  const int nc = flat_ncomp(tmpl);
  agp_kernel_component comps[AGP_MAX_COMPONENTS];
  const int64_t cbase = 4 + ns + (int64_t)M * D + M + (int64_t)M * M;
  if (nc > 0) {
    for (int i = 0; i < nc; i++) {
      comps[i].kind = tmpl->kernel.components[i].kind;
      comps[i].variance = f[cbase + i];
      comps[i].inv_lengthscale = f[cbase + nc + i];
    }
    p.kernel.components = comps;
  }
  if (!flat_grad) return agp_svgp_elbo(c, ds, offset, count, &p, num_data, global_batch, elbo_out);
  double* g = flat_grad;
  agp_svgp_grads go{};
  go.dvariance = g;
  go.dinv_lengthscale = g + 1;
  go.dlinear_c = g + 1 + ns;
  go.dmean_const = g + 2 + ns;
  go.dlik_sigma2 = g + 3 + ns;
  go.dZ = g + 4 + ns;
  go.dm = go.dZ + (int64_t)M * D;
  go.dLq = go.dm + M;
  if (nc > 0) {
    go.dcomp_variance = g + cbase;
    go.dcomp_inv_lengthscale = g + cbase + nc;
  }
  return agp_svgp_elbo_grad(c, ds, offset, count, &p, num_data, global_batch, elbo_out, &go);
}

extern "C" int32_t agp_svgp_elbo(agp_ctx* c, agp_dataset* ds, int64_t offset, int64_t count, const agp_svgp_params* p,
                                 double num_data, int64_t global_batch, double* elbo_out) {
  const int32_t s = agp_svgp_sweep(c, ds, offset, count, p, num_data, global_batch, 0);
  if (s != AGP_OK) {
    if (c && !(c->comm && c->nranks > 1 && global_batch <= 0)) signal_failure_to_peers(c, p, false);
    return s;
  }
  OK(allreduce_if_needed(c));
  return agp_svgp_finish(c, elbo_out, nullptr);
}

extern "C" int32_t agp_svgp_prior_kl(agp_ctx* c, const agp_svgp_params* p, double* kl_out) {
  if (!c || !p || !kl_out) return fail(AGP_ERR_INVALID, "agp_svgp_prior_kl: NULL argument");
  OK(prepare_step(c, p));
  OK(run_kl(c, c->small.p));
  CU(cudaMemcpyAsync(kl_out, c->small.p, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  return check_step_flags(c, false);
}

extern "C" int32_t agp_svgp_posterior(agp_ctx* c, const agp_svgp_params* p, double* Lk_out, double* B_out, double* alpha_out) {
  if (!c || !p) return fail(AGP_ERR_INVALID, "agp_svgp_posterior: NULL argument");
  OK(prepare_step(c, p));
  SvgpState& st = c->st;
  const int M = st.M, Mp = st.Mp;
  if (alpha_out) {
    // alpha = Lk^-T mt   (NonCentered: Lk' \ m, SVA.jl:182; Centered: Kuu \ (m - mean(fz)), SVA.jl:133)
    vec_to_rhs_kernel<<<(Mp * 64 + 255) / 256, 256, 0, c->stream>>>(c->mt.p, 0.0, Mp, Mp, c->vec64.p);
    LAUNCHED(c);
    KCHECK();
    OK(solve_lk<TR_RHS_BWD>(c, c->vec64.p, 64, 1));
    rhs_to_vec_kernel<<<(Mp + 255) / 256, 256, 0, c->stream>>>(c->vec64.p, Mp, c->vec64b.p);
    LAUNCHED(c);
    KCHECK();
    CU(cudaMemcpyAsync(alpha_out, c->vec64b.p, sizeof(double) * M, cudaMemcpyDeviceToHost, c->stream));
  }
  if (Lk_out) CU(cudaMemcpy2DAsync(Lk_out, sizeof(double) * M, c->Lk.p, sizeof(double) * Mp, sizeof(double) * M, M, cudaMemcpyDeviceToHost, c->stream));
  if (B_out) CU(cudaMemcpy2DAsync(B_out, sizeof(double) * M, c->Bt_cm.p, sizeof(double) * Mp, sizeof(double) * M, M, cudaMemcpyDeviceToHost, c->stream));
  return check_step_flags(c, false);
}

extern "C" int32_t agp_svgp_mean_and_var(agp_ctx* c, const agp_svgp_params* p, const double* Xnew, int64_t n, double* mu_out,
                                         double* var_out) {
  if (!c || !p || !Xnew || n < 1) return fail(AGP_ERR_INVALID, "agp_svgp_mean_and_var: bad arguments");
  OK(prepare_step(c, p));
  SvgpState& st = c->st;
  st.scale = 1.0;
  const int D = st.D;
  OK(c->mu_out.ensure(n + BN));
  OK(c->var_out.ensure(n + BN));
  DevBuf xbuf;
  OK(xbuf.ensure((n + BN) * D));
  CU(cudaMemcpyAsync(xbuf.p, Xnew, sizeof(double) * n * D, cudaMemcpyHostToDevice, c->stream));
  int32_t s = sweep_points(c, xbuf.p, nullptr, n, false, true, c->mu_out.p, c->var_out.p);
  if (s == AGP_OK) {
    if (mu_out) cudaMemcpyAsync(mu_out, c->mu_out.p, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream);
    if (var_out) cudaMemcpyAsync(var_out, c->var_out.p, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream);
  }
  cudaError_t e = cudaStreamSynchronize(c->stream);
  xbuf.release();
  if (s != AGP_OK) return s;
  if (e != cudaSuccess) return fail(AGP_ERR_CUDA, "mean_and_var: %s", cudaGetErrorString(e));
  return check_step_flags(c, false);
}

// ---------------------------------------------------------------------------------------------------
// SVGP: full (cross-)covariance of the approximate posterior
// ---------------------------------------------------------------------------------------------------
// A = Lk^-1 Kuf and C = Bt^T A for one set of points (single chunk), into the given scratch matrices.
static int32_t project_points(agp_ctx* c, const double* X_dev, int n, int ncols, double* Abuf, double* Cbuf, int64_t ldc) {
  SvgpState& st = c->st;
  OK(launch_s1(c, s1_args(c, Abuf, ldc, X_dev, n), ncols / BN));
  EpiS2 e2{Cbuf, ldc, c->scc_part.p, ldc};
  OK((run_gemm<A_KM, B_KN>(c, st.nb, ncols / BN, c->Bt_rm.p, st.Mp, Abuf, ldc, st.Mp, KR_UPPER, TS_ALL, e2)));
  return AGP_OK;
}

constexpr int64_t AGP_MAX_COV_POINTS = 16384;

extern "C" int32_t agp_svgp_mean_and_cov(agp_ctx* c, const agp_svgp_params* p, const double* X1, int64_t n1, const double* X2, int64_t n2,
                                         double* mu1_out, double* cov_out) {
  if (!c || !p || !X1 || n1 < 1 || !cov_out) return fail(AGP_ERR_INVALID, "agp_svgp_mean_and_cov: bad arguments");
  const bool cross = X2 != nullptr;
  if (!cross) n2 = n1;
  if (n2 < 1) return fail(AGP_ERR_INVALID, "agp_svgp_mean_and_cov: bad arguments");
  if (n1 > AGP_MAX_COV_POINTS || n2 > AGP_MAX_COV_POINTS)
    return fail(AGP_ERR_UNSUPPORTED, "full covariances are limited to %lld points per argument (the matrix is dense)", (long long)AGP_MAX_COV_POINTS);
  OK(prepare_step(c, p));
  SvgpState& st = c->st;
  st.scale = 1.0;
  const int D = st.D, Mp = st.Mp;
  const int n1p = (int)round_up(n1, BM), n2p = (int)round_up(n2, BM);
  OK(ensure_sweep_workspace(c, std::max(n1p, n2p), true));
  const int64_t ldc = c->chunk_cols;
  OK(c->px1.ensure((int64_t)n1p * D));
  OK(c->pxs1.ensure((int64_t)n1p * D));
  OK(c->pxn1.ensure(n1p));
  OK(c->pcov.ensure((int64_t)n1p * n2p));
  OK(c->mu_out.ensure(n1p));
  OK(c->var_out.ensure(n1p));
  CU(cudaMemsetAsync(c->px1.p, 0, sizeof(double) * n1p * D, c->stream));
  CU(cudaMemcpyAsync(c->px1.p, X1, sizeof(double) * n1 * D, cudaMemcpyHostToDevice, c->stream));
  KernelParams kx = st.kp;
  kx.M = (int)n1;
  prep_z_kernel<<<(n1p + 127) / 128, 128, 0, c->stream>>>(c->px1.p, c->pxs1.p, c->pxn1.p, nullptr, n1p, kx);
  LAUNCHED(c);
  KCHECK();
  OK(project_points(c, c->px1.p, (int)n1, n1p, c->A.p, c->C.p, ldc));
  if (mu1_out) {
    // the per-point stage of the sweep in prediction mode; project_points ran S2 on DMMA
    OK(sweep_s3(c, SweepPlan{}, c->px1.p, nullptr, 0, (int)n1, n1p, true, c->mu_out.p, c->var_out.p, nullptr));
    CU(cudaMemcpyAsync(mu1_out, c->mu_out.p, sizeof(double) * n1, cudaMemcpyDeviceToHost, c->stream));
  }
  const double *A2 = c->A.p, *C2 = c->C.p;
  if (cross) {
    OK(c->px2.ensure((int64_t)n2p * D));
    OK(c->pxs2.ensure((int64_t)n2p * D));
    OK(c->pxn2.ensure(n2p));
    CU(cudaMemsetAsync(c->px2.p, 0, sizeof(double) * n2p * D, c->stream));
    CU(cudaMemcpyAsync(c->px2.p, X2, sizeof(double) * n2 * D, cudaMemcpyHostToDevice, c->stream));
    KernelParams ky = st.kp;
    ky.M = (int)n2;
    prep_z_kernel<<<(n2p + 127) / 128, 128, 0, c->stream>>>(c->px2.p, c->pxs2.p, c->pxn2.p, nullptr, n2p, ky);
    LAUNCHED(c);
    KCHECK();
    OK(project_points(c, c->px2.p, (int)n2, n2p, c->Ab.p, c->As.p, ldc));
    A2 = c->Ab.p;
    C2 = c->As.p;
    cross_k_kernel<<<dim3((n1p + 127) / 128, n2p), 128, 0, c->stream>>>(c->pcov.p, n1p, c->pxs1.p, c->pxn1.p, (int)n1, c->pxs2.p, c->pxn2.p, (int)n2, n1p, st.kp);
  } else {
    // cov(f.prior, x): the one-argument kernelmatrix (exactly zero distances on the diagonal)
    build_kuu_kernel<<<dim3((n1p + 127) / 128, n1p), 128, 0, c->stream>>>(c->pcov.p, n1p, c->pxs1.p, c->pxn1.p, 0.0, kx);
  }
  LAUNCHED(c);
  KCHECK();
  // cov = K - A1^T A2 + C1^T C2   (SVA.jl:227 / :263)
  OK((run_gemm<A_KM, B_KN>(c, n1p / BM, n2p / BN, c->A.p, ldc, A2, ldc, Mp, KR_FULL, TS_ALL, epi_store(c->pcov.p, n1p, false, -1.0, 1.0))));
  OK((run_gemm<A_KM, B_KN>(c, n1p / BM, n2p / BN, c->C.p, ldc, C2, ldc, Mp, KR_FULL, TS_ALL, epi_store(c->pcov.p, n1p, false, 1.0, 1.0))));
  CU(cudaMemcpy2DAsync(cov_out, sizeof(double) * n1, c->pcov.p, sizeof(double) * n1p, sizeof(double) * n1, n2, cudaMemcpyDeviceToHost, c->stream));
  return check_step_flags(c, false);
}

// ---------------------------------------------------------------------------------------------------
// prior covariance matrices and the in-run FP64 peak measurement
// ---------------------------------------------------------------------------------------------------
extern "C" int32_t agp_kernel_matrix(agp_ctx* c, const agp_kernel* k, int32_t D, const double* X1, int64_t n1, const double* X2, int64_t n2,
                                     double* K_out) {
  if (!c || !k || !X1 || !K_out || n1 < 1 || D < 1) return fail(AGP_ERR_INVALID, "agp_kernel_matrix: bad arguments");
  if (D > MAXD) return fail(AGP_ERR_UNSUPPORTED, "input dimension %d > %d is not supported on device", D, MAXD);
  const bool cross = X2 != nullptr;
  if (!cross) n2 = n1;
  if (n2 < 1 || n1 > AGP_MAX_COV_POINTS || n2 > AGP_MAX_COV_POINTS) return fail(AGP_ERR_INVALID, "agp_kernel_matrix: 1 <= n <= %lld", (long long)AGP_MAX_COV_POINTS);
  CU(cudaSetDevice(c->device));
  KernelParams kp;
  OK(fill_kernel_params(k, D, 0, kp));
  OK(c->px1.ensure(n1 * D));
  OK(c->pxs1.ensure(n1 * D));
  OK(c->pxn1.ensure(n1));
  OK(c->pcov.ensure(n1 * n2));
  CU(cudaMemcpyAsync(c->px1.p, X1, sizeof(double) * n1 * D, cudaMemcpyHostToDevice, c->stream));
  kp.M = (int)n1;
  prep_z_kernel<<<(int)((n1 + 127) / 128), 128, 0, c->stream>>>(c->px1.p, c->pxs1.p, c->pxn1.p, nullptr, (int)n1, kp);
  LAUNCHED(c);
  KCHECK();
  if (cross) {
    OK(c->px2.ensure(n2 * D));
    OK(c->pxs2.ensure(n2 * D));
    OK(c->pxn2.ensure(n2));
    CU(cudaMemcpyAsync(c->px2.p, X2, sizeof(double) * n2 * D, cudaMemcpyHostToDevice, c->stream));
    KernelParams ky = kp;
    ky.M = (int)n2;
    prep_z_kernel<<<(int)((n2 + 127) / 128), 128, 0, c->stream>>>(c->px2.p, c->pxs2.p, c->pxn2.p, nullptr, (int)n2, ky);
    LAUNCHED(c);
    KCHECK();
    cross_k_kernel<<<dim3((int)((n1 + 127) / 128), (int)n2), 128, 0, c->stream>>>(c->pcov.p, n1, c->pxs1.p, c->pxn1.p, (int)n1, c->pxs2.p, c->pxn2.p, (int)n2, (int)n1, kp);
  } else {
    build_kuu_kernel<<<dim3((int)((n1 + 127) / 128), (int)n1), 128, 0, c->stream>>>(c->pcov.p, (int)n1, c->pxs1.p, c->pxn1.p, 0.0, kp);
  }
  LAUNCHED(c);
  KCHECK();
  CU(cudaMemcpyAsync(K_out, c->pcov.p, sizeof(double) * n1 * n2, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return AGP_OK;
}

// FP64 issue-rate microbenchmarks (the roofline denominators bench.py prints next to every FP64 fraction): register-resident
// DMMA.8x8x4 chains (8 independent accumulators per warp) and DFMA chains (8 per thread), 1024 threads x 2 blocks per SM.
__global__ void __launch_bounds__(1024) peak_dmma_kernel(double* out, int iters, double s) {
  double acc[8][2];  // 8 independent accumulators per warp: 37.1 TFLOP/s on B200; 16 measure lower (28.6, profiles/r01_fp64_peak.jsonl)
#pragma unroll
  for (int i = 0; i < 8; i++) acc[i][0] = acc[i][1] = 0.0;
  const double a = s + threadIdx.x * 1e-12, b = 1e-3 * s;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) dmma884(acc[i], a, b);
  }
  double r = 0.0;
#pragma unroll
  for (int i = 0; i < 8; i++) r += acc[i][0] + acc[i][1];
  out[blockIdx.x * (int64_t)blockDim.x + threadIdx.x] = r;
}
__global__ void __launch_bounds__(1024) peak_dfma_kernel(double* out, int iters, double s) {
  double acc[8];
#pragma unroll
  for (int i = 0; i < 8; i++) acc[i] = threadIdx.x * 1e-9 + i;
  const double a = s, b = 1.0 - s;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = fma(acc[i], a, b);
  }
  double r = 0.0;
#pragma unroll
  for (int i = 0; i < 8; i++) r += acc[i];
  out[blockIdx.x * (int64_t)blockDim.x + threadIdx.x] = r;
}
extern "C" int32_t agp_fp64_peak(agp_ctx* c, int32_t which, double* tflops_out) {
  if (!c || !tflops_out || which < 0 || which > 1) return fail(AGP_ERR_INVALID, "agp_fp64_peak: bad arguments");
  CU(cudaSetDevice(c->device));
  const int threads = 1024, blocks = 2 * c->sms, iters = 20000;
  OK(c->pcov.ensure((int64_t)threads * blocks));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 4; rep++) {  // rep 0 warms up the clocks
    CU(cudaEventRecord(e0, c->stream));
    if (which == 0) peak_dmma_kernel<<<blocks, threads, 0, c->stream>>>(c->pcov.p, iters, 0.5);
    else peak_dfma_kernel<<<blocks, threads, 0, c->stream>>>(c->pcov.p, iters, 0.5);
    LAUNCHED(c);
    CU(cudaEventRecord(e1, c->stream));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    if (rep > 0) best = std::min(best, ms);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  KCHECK();
  const double flop = which == 0 ? 2.0 * 256 * 8 * (double)iters * (threads / 32) * blocks : 2.0 * 8 * (double)iters * threads * blocks;
  *tflops_out = flop / (best * 1e-3) / 1e12;
  return AGP_OK;
}

#include "small_host.inc"
#include "laplace_host.inc"
