// Shared definitions for the basq_b200 CUDA library (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/basq_b200.h"

namespace basq {

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);

#define BASQ_CUDA(expr)                                                                   \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      basq::set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr,               \
                      cudaGetErrorString(_e));                                            \
      return BASQ_ERR_CUDA;                                                               \
    }                                                                                     \
  } while (0)

#define BASQ_CHECK(cond, code, ...)                                                       \
  do {                                                                                    \
    if (!(cond)) {                                                                        \
      basq::set_error(__VA_ARGS__);                                                       \
      return (code);                                                                      \
    }                                                                                     \
  } while (0)

#define BASQ_TRY(expr)                                                                    \
  do {                                                                                    \
    int _s = (expr);                                                                      \
    if (_s != BASQ_OK) return _s;                                                         \
  } while (0)

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
enum Phase { PH_PREP = 0, PH_SETSUM = 1, PH_PROJ = 2, PH_CAR = 3, PH_APPLY = 4, PH_NYS = 5, PH_GP = 6, PH_OTHER = 7, PH_COUNT = 8 };

}  // namespace basq

struct basq_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  // Private block cache for the library's scratch (DevBuf below): a freed block goes onto a free list and is
  // handed out again to the next request of the same size class, whole - blocks are never split or merged.
  // Everything the library launches runs on `stream`, so a block may be reused without a fence.  In steady
  // state no allocation reaches the driver.  (Round 2 first used a cudaMemPool_t here: its best-fit carving
  // of free blocks made the layout depend on the order of requests, and a call sequence that differed from
  // the warmed-up one - the host-buffer entry after device-resident calls, the next leg of the bench - ran
  // into re-mapping stalls of 0.15-1.65 s per call.)  basq_ctx_trim / the end of every top-level call
  // release everything above pool_keep bytes (default: keep all).
  struct Block { void* p; size_t bytes; };
  std::vector<Block> free_blocks;
  size_t cached_bytes = 0;          // on the free list
  size_t live_bytes = 0;            // handed out
  int64_t driver_allocs = 0;
  uint64_t pool_keep = 0;
  static size_t size_class(size_t n) {
    if (n < 4096) n = 4096;
    size_t p2 = 4096;
    while (p2 * 2 <= n) p2 *= 2;
    const size_t gran = p2 / 8 < 4096 ? 4096 : p2 / 8;       // at most 12.5 % above the request
    return (n + gran - 1) / gran * gran;
  }
  // returns nullptr when the device is out of memory even after the cache was emptied
  void* block_alloc(size_t n, size_t* got) {
    const size_t cls = size_class(n);
    int best = -1;
    for (int i = 0; i < (int)free_blocks.size(); ++i)
      if (free_blocks[i].bytes >= cls && free_blocks[i].bytes <= cls + cls / 4 &&
          (best < 0 || free_blocks[i].bytes < free_blocks[best].bytes))
        best = i;
    void* p = nullptr;
    if (best >= 0) {
      p = free_blocks[best].p;
      *got = free_blocks[best].bytes;
      cached_bytes -= *got;
      free_blocks[best] = free_blocks.back();
      free_blocks.pop_back();
    } else {
      if (cudaMalloc(&p, cls) != cudaSuccess) {
        (void)cudaGetLastError();
        block_trim(0);
        if (cudaMalloc(&p, cls) != cudaSuccess) {
          (void)cudaGetLastError();
          return nullptr;
        }
      }
      ++driver_allocs;
      *got = cls;
    }
    live_bytes += *got;
    return p;
  }
  void block_free(void* p, size_t bytes) {
    free_blocks.push_back({p, bytes});
    cached_bytes += bytes;
    live_bytes -= bytes;
  }
  // hand cached blocks back to the driver, largest first, until at most `keep` bytes stay cached
  void block_trim(size_t keep) {
    if (cached_bytes <= keep) return;
    cudaStreamSynchronize(stream);   // queued work may still use a block that is already on the free list
    while (cached_bytes > keep && !free_blocks.empty()) {
      int big = 0;
      for (int i = 1; i < (int)free_blocks.size(); ++i)
        if (free_blocks[i].bytes > free_blocks[big].bytes) big = i;
      cudaFree(free_blocks[big].p);
      cached_bytes -= free_blocks[big].bytes;
      free_blocks[big] = free_blocks.back();
      free_blocks.pop_back();
    }
    (void)cudaGetLastError();
  }
  int num_sms = 0;
  size_t smem_optin = 0;
  int64_t launches = 0;
  int64_t pair_evals = 0;
  bool profile = false;
  int timer_depth = 0;
  bool force_general_car = false;  // BASQ_CAR_GENERAL=1: always use the global-memory kernel (tests)
  bool no_gpvar = false;           // BASQ_GPVAR=0: chunked fp64-GEMM posterior variance for fp32 inputs too (A/B)
  // per-context driver objects that are expensive to create per call (api.cu): pinned staging ring of the level
  // calls, side stream + events of basq_recombine_host
  static constexpr int STAGE_SLOTS = 8;
  unsigned char* stage = nullptr;
  size_t stage_slot_bytes = 0;
  cudaEvent_t stage_ev[STAGE_SLOTS] = {nullptr};
  int stage_next = 0;
  cudaStream_t side = nullptr;
  // candidate buffer of basq_recombine_host, kept between calls and outside the pool: carving 400 MB out of the
  // pool's free blocks before every other request reshuffles them from call to call (observed: steps of
  // 127-245 ms and an occasional second of re-growth where the device-resident path takes a steady 125 ms)
  void* host_x = nullptr;
  size_t host_x_bytes = 0;
  // basq_ctx_stage_candidates: what currently travels / sits in host_x for basq_session_create_staged
  int64_t staged_N = -1;
  int staged_d = 0, staged_dtype = 0;
  double* staged_mu = nullptr;
  cudaEvent_t side_ev[2] = {nullptr, nullptr};
  bool eval_f32 = false;           // basq_ctx_allow_f32_eval: fp64 inputs may be evaluated on the fp32 tensor-core path
  bool reproducible = false;       // basq_ctx_reproducible: sessions sum on a grid, the same bits for any split over ranks
  int64_t demotions = 0;
  uint64_t seed = 0;               // basq_ctx_set_seed: key of the library's own Gaussian draws (Nystrom test matrix)
  uint64_t draws = 0;              // test matrices drawn since the seed was set (each call uses key seed + draws)
  bool no_nlsum = false;           // BASQ_NLSUM=0: chunked fp64-GEMM path for the non-linear modes in fp32 too (A/B)
  // fp32 inputs are promoted to the fp64 path when max_m |(K_ZX W)_m|_1 exceeds kappa_max (api.cu:
  // session_create_impl); BASQ_F32_KAPPA_MAX overrides, 0 disables
  double kappa_max = 64.0;
  double last_kappa = 0.0;
  int64_t promotions = 0;
  bool trace = false;      // BASQ_TRACE=1: wall-clock trace points on stderr (synchronising)
  double trace_t0 = 0.0;
  double phase_ms[basq::PH_COUNT] = {0};
  int64_t phase_calls[basq::PH_COUNT] = {0};
  // phase spans recorded since the last read: (phase, start event, stop event); events come from a
  // free list so that profiling never synchronises inside the timed region
  struct Span { int phase; cudaEvent_t e0, e1; };
  std::vector<Span> spans;
  std::vector<cudaEvent_t> free_events;
  cudaEvent_t take_event() {
    if (!free_events.empty()) { cudaEvent_t e = free_events.back(); free_events.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
  }
  // fold finished spans into phase_ms / phase_calls (synchronises the stream)
  void resolve_spans() {
    if (spans.empty()) return;
    cudaStreamSynchronize(stream);
    for (const Span& s : spans) {
      float ms = 0.f;
      if (s.e0 && s.e1 && cudaEventElapsedTime(&ms, s.e0, s.e1) == cudaSuccess) {
        phase_ms[s.phase] += ms;
        phase_calls[s.phase] += 1;
      }
      if (s.e0) free_events.push_back(s.e0);
      if (s.e1) free_events.push_back(s.e1);
    }
    spans.clear();
    (void)cudaGetLastError();
  }
};

namespace basq {

// RAII phase timer (only active when ctx->profile): records a start/stop event pair on the context's
// stream without synchronising; basq_ctx_profile_read resolves them.  Nested timers are ignored.
// Every outermost phase is also an NVTX range ("basq:<phase>", visible to Nsight Systems / ncu --nvtx).
static inline const char* phase_name(int ph) {
  static const char* const names[PH_COUNT] = {"basq:prepare", "basq:set_sum", "basq:projection", "basq:caratheodory",
                                              "basq:apply", "basq:nystrom", "basq:gp_predict", "basq:other"};
  return (ph >= 0 && ph < PH_COUNT) ? names[ph] : "basq:?";
}
struct PhaseTimer {
  basq_ctx* ctx;
  int phase;
  bool active;
  bool outer;
  cudaEvent_t e0 = nullptr;
  PhaseTimer(basq_ctx* c, int ph) : ctx(c), phase(ph) {
    outer = (ctx->timer_depth++ == 0);
    if (outer) nvtxRangePushA(phase_name(ph));
    active = outer && ctx->profile;
    if (active) {
      e0 = ctx->take_event();
      cudaEventRecord(e0, ctx->stream);
    }
  }
  ~PhaseTimer() {
    ctx->timer_depth--;
    if (outer) nvtxRangePop();
    if (active) {
      cudaEvent_t e1 = ctx->take_event();
      cudaEventRecord(e1, ctx->stream);
      ctx->spans.push_back({phase, e0, e1});
    }
  }
};

// Device buffer with RAII from the context's block cache (basq_ctx::block_alloc): in steady state neither
// alloc nor release reaches the driver or synchronises the device - the round loop allocates and frees scratch
// every round.  Everything the library launches runs on the context's one stream, so a released block may be
// handed to the next allocation without a fence.
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;      // size of the cache block behind p (>= the request)
  basq_ctx* owner = nullptr;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p && owner) owner->block_free(p, bytes);
    p = nullptr;
    bytes = 0;
  }
  int alloc(basq_ctx* ctx, size_t n) {
    release();
    if (n == 0) n = 16;
    owner = ctx;
    p = ctx->block_alloc(n, &bytes);
    if (!p) {
      set_error("device allocation of %zu bytes failed (%zu bytes live in this context)", n, ctx->live_bytes);
      bytes = 0;
      return BASQ_ERR_CUDA;
    }
    return BASQ_OK;
  }
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

// wall-clock trace point (debug aid; synchronises the stream when enabled)
void trace_point(basq_ctx* ctx, const char* label);

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------------------------
// kernel parameters in device-friendly form
// ---------------------------------------------------------------------------------------------
// fp32 evaluation uses the expansion  arg = a_x + b_z + sum_i x'_i * zz_i  on centred, scaled
// coordinates (the same form gpytorch/torch.cdist use):
//   RBF    : x' = (x-c) * sqrt(log2(e)/2) / l ; a_x = -|x'|^2 ; b_z = -|z'|^2 + log2(os) ; zz = 2 z'
//            k  = exp2(arg)
//   Matern : x' = (x-c) / l ; a_x = |x'|^2 ; b_z = |z'|^2 ; zz = -2 z' ; r^2 = max(arg, 0)
// fp64 evaluation uses direct differences on x' = (x-c)/l.
struct KParams {
  int family;
  int d;
  int dp;  // padded dimension used by the compiled kernels
  double outputscale;
  float log2_os;
  float os_f;
  float scale_f[BASQ_MAX_DIM];   // fp32 per-dim multiplier (includes the RBF sqrt(log2e/2))
  double scale_d[BASQ_MAX_DIM];  // 1 / lengthscale
  double center[BASQ_MAX_DIM];
};

// padded dimensions that have compiled instantiations
static inline int padded_dim(int d) {
  const int opts[] = {2, 4, 6, 8, 10, 12, 16, 20, 24, 32};
  for (int o : opts)
    if (d <= o) return o;
  return -1;
}

// ---------------------------------------------------------------------------------------------
// candidate record (array of structs; what each Tchernychova-Lyons round streams)
//   f32: [ wf:f64 | mu:f64 | idx:i32 | a:f32 | x'[DP]:f32 ]  padded to 16 B   (64 B at DP = 10)
//   f64: [ wf:f64 | mu:f64 | idx:i64 | x'[DP]:f64 ]          padded to 16 B
// wf is the weight the feature sums use (mu, or mu * m(x) for WSABI-L; the per-point factor itself
// for the non-linear modes), mu the plain measure weight (set masses, final answer).
// ---------------------------------------------------------------------------------------------
__host__ __device__ static inline int rec_bytes_f32(int dp) { return ((24 + 4 * dp) + 15) / 16 * 16; }
__host__ __device__ static inline int rec_bytes_f64(int dp) { return ((24 + 8 * dp) + 15) / 16 * 16; }

// non-linearity applied per (landmark, point) pair before accumulation
enum NlMode { NL_LIN = 0, NL_WSABIM = 1, NL_MMLT = 2 };

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// exact float -> double for non-negative finite floats without touching the conversion pipe
// (zero maps to 2^-127, which is below anything the sums can resolve).
__device__ __forceinline__ double f2d_pos(float k) {
  unsigned u = __float_as_uint(k);
  return __hiloint2double((int)((u >> 3) + 0x38000000u), (int)(u << 29));
}

// Reproducible mode, host side: the grids of sums of at most R terms whose |sum| is bounded by B.  gm = 1.5 * 2^52 Q
// with Q = 2^(ceil(log2 B) - 51) (every term below 2^51 Q, every partial sum below 2^53 Q); gm2 the grid of the
// remainders term - hi, each below Q / 2, so their sum is below R Q / 2.  B must be finite and below 2^1000.
inline void grid_pair(double B, double R, double* gm, double* gm2) {
  int e = -1000;
  if (B > 0.0) frexp(B, &e);                 // B <= 2^e
  e = e < -800 ? -800 : e;
  *gm = ldexp(1.5, e - 51 + 52);
  int e2 = 0;
  frexp(R * ldexp(0.5, e - 51), &e2);        // R Q / 2 <= 2^e2
  *gm2 = ldexp(1.5, e2 - 51 + 52);
}

// Reproducible mode: the term a * b rounded to the grid Q of gm = 1.5 * 2^52 * Q (exact for |a b| < 2^51 Q: gm + a b
// then lies in [2^52 Q, 2^53 Q), where the spacing of doubles is Q).  Sums of such terms are multiples of Q and
// exact while they stay below 2^53 Q, so they do not depend on the order of the additions, on the tiling or on
// how the terms are split over ranks and all-reduced.
__device__ __forceinline__ double grid_round(double a, double b, double gm) { return __dsub_rn(__fma_rn(a, b, gm), gm); }

// One kernel evaluation in fp32 from prepared operands.  Every fp32 kernel in the library goes
// through the same operation sequence (acc = a + b; acc = fma(x_i, zz_i, acc) for i ascending;
// finish_f32) with the same operand roles, so k(z, x) is bit-identical wherever it is recomputed
// (set sums of every round, features, Gram matrices).
__device__ __forceinline__ float finish_f32(int fam, float acc, float os_f) {
  if (fam == BASQ_RBF) {
    return ex2_approx(acc);
  } else {
    const float r2 = fmaxf(acc, 0.f);
    const float r = sqrt_approx(r2);
    if (fam == BASQ_MATERN15) {
      const float c = 1.7320508075688772f;
      const float e = ex2_approx(__fmul_rn(-c * 1.4426950408889634f, r));
      return __fmul_rn(__fmul_rn(os_f, __fmaf_rn(c, r, 1.f)), e);
    } else {
      const float c = 2.23606797749979f;
      const float e = ex2_approx(__fmul_rn(-c * 1.4426950408889634f, r));
      const float poly = __fmaf_rn(1.6666666666666667f, r2, __fmaf_rn(c, r, 1.f));
      return __fmul_rn(__fmul_rn(os_f, poly), e);
    }
  }
}

template <int FAM, int DP>
__device__ __forceinline__ float pair_eval_f32(const float* __restrict__ x, float a, const float* __restrict__ zz,
                                               float b, float os_f) {
  float acc = __fadd_rn(a, b);
#pragma unroll
  for (int i = 0; i < DP; ++i) acc = __fmaf_rn(x[i], zz[i], acc);
  return finish_f32(FAM, acc, os_f);
}

__device__ __forceinline__ double finish_f64(int fam, double r2, double os) {
  if (fam == BASQ_RBF) {
    return os * exp(-0.5 * r2);
  } else {
    const double r = sqrt(r2);
    if (fam == BASQ_MATERN15) {
      const double c = 1.7320508075688772;
      return os * (1.0 + c * r) * exp(-c * r);
    } else {
      const double c = 2.23606797749979;
      return os * (1.0 + c * r + (5.0 / 3.0) * r2) * exp(-c * r);
    }
  }
}

template <int FAM, int DP>
__device__ __forceinline__ double pair_eval_f64(const double* __restrict__ x, const double* __restrict__ z, double os) {
  double r2 = 0.0;
#pragma unroll
  for (int i = 0; i < DP; ++i) {
    const double df = x[i] - z[i];
    r2 = fma(df, df, r2);
  }
  return finish_f64(FAM, r2, os);
}

__device__ __forceinline__ double nl_apply(int nl, double c, double sz, double sx) {
  if (nl == NL_WSABIM) return sz * c * sx + 0.5 * c * c;
  if (nl == NL_MMLT) return sz * sx * expm1(c);
  return c;
}
#endif  // __CUDACC__

// ---------------------------------------------------------------------------------------------
// prepared landmark set (device arrays)
// ---------------------------------------------------------------------------------------------
struct LmView {
  const void* zz = nullptr;  // f32: [count, dp] floats (2z' / -2z') ; f64: [count, dp] doubles (z')
  const float* b = nullptr;  // f32: [count] floats
  const float* lmA = nullptr;  // f32, whole-set views only: tile-blocked tensor-core operand (setsum_mma.cuh)
  int count = 0;
  int dp = 0;
  int dtype = BASQ_F32;
};

struct Landmarks {
  int count = 0;
  int dp = 0;
  int dtype = BASQ_F32;
  DevBuf zz;
  DevBuf b;
  DevBuf lmA;
  void release() {
    zz.release();
    b.release();
    lmA.release();
  }
  LmView view(int first = 0, int cnt = -1) const {
    LmView v;
    if (cnt < 0) cnt = count - first;
    if (first == 0 && cnt == count && dtype == BASQ_F32) v.lmA = lmA.as<float>();
    const size_t esz = dtype == BASQ_F32 ? 4 : 8;
    v.zz = (const unsigned char*)zz.p + (size_t)first * dp * esz;
    v.b = dtype == BASQ_F32 ? b.as<float>() + first : nullptr;
    v.count = cnt;
    v.dp = dp;
    v.dtype = dtype;
    return v;
  }
};

// ---------------------------------------------------------------------------------------------
// internal entry points (one per translation unit)
// ---------------------------------------------------------------------------------------------
// kparams.cu
int make_kparams(const basq_kernel_desc* desc, KParams* kp);
int compute_center(basq_ctx* ctx, const basq_kernel_desc* desc, const void* Z, int64_t M, KParams* kp);
int prep_landmarks(basq_ctx* ctx, const KParams& kp, int dtype, const void* Z0, int64_t M0, const void* Z1,
                   int64_t M1, Landmarks* out);

// gram.cu
// out[a, b] fp64 row-major (ld = ldo): base kernel between prepared landmarks and raw points P[b, d]
int base_gram(basq_ctx* ctx, const KParams& kp, const LmView& lm, const void* P, int64_t b, double* out,
              int64_t ldo);
// same, the points being live records [p_lo, p_hi) of a pool (already scaled coordinates)
struct RecPool;
int base_gram_records(basq_ctx* ctx, const KParams& kp, const LmView& lm, const RecPool& pool, int64_t p_lo,
                      int64_t p_hi, double* out, int64_t ldo);
// mean_out[N] = c0 + sum_o coef[o] k(lm_o, x)   (fp64 accumulation)
int landmark_dot(basq_ctx* ctx, const KParams& kp, const LmView& lm, const double* coef, double c0,
                 const void* P, int64_t N, double* out);
// out[p] = c0 + sum_{j < cols} G[p, j]   (p < n; fixed order)
int rowsum_cols(basq_ctx* ctx, const double* G, int64_t n, int cols, double c0, double* out);
// whether gp_predict_impl computes the variance on the tensor cores (gp_variance_tc): fp32 inputs, unless
// BASQ_GPVAR=0 selects the chunked fp64-GEMM route
bool gpvar_route(basq_ctx* ctx, const basq_kernel_desc* desc);
int gp_predict_impl(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const LmView& lmobs,
                    const void* X, int64_t N, double* mean_out, double* var_out);
// per-point / per-landmark factor of the warped kernels (m(x) or mu_g(x)); out == nullptr allowed
int warp_factor(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const LmView& lmobs,
                const void* X, int64_t N, double* out);

// records.cu
struct RecPool {
  int dtype = BASQ_F32;
  int dp = 0;
  int rec_bytes = 0;
  DevBuf buf[2];
  int cur = 0;
  int64_t count = 0;
  int64_t capacity = 0;
};
// round_buffer: also allocate the second buffer that apply_round compacts into (recombination only)
int build_records(basq_ctx* ctx, const KParams& kp, int dtype, const void* X, int64_t N, double uniform_w,
                  const double* mu, const double* factor, bool factor_in_weight, RecPool* pool,
                  bool round_buffer = true);
// grid_m != 0: reproducible sums, every term rounded to the grid of grid_m (grid_round)
// (masses and objective terms are fp64: the remainders of the terms go to the grid of grid_m2, summed into *_out2)
int set_masses(basq_ctx* ctx, const RecPool& pool, int64_t off_glob, int S, int S_eff, double* mass_out,
               double grid_m = 0.0, double grid_m2 = 0.0, double* mass_out2 = nullptr);
int cell_objective(basq_ctx* ctx, const RecPool& pool, int64_t off_glob, int S, int S_eff, const double* obj,
                   double* out, double grid_m = 0.0, double grid_m2 = 0.0, double* out2 = nullptr);
// max_host[3] = maxima over the live records of |wf|, |mu| and |mu obj[idx]| (obj may be NULL); synchronises
int record_maxima(basq_ctx* ctx, const RecPool& pool, const double* obj, double* max_host);
int apply_round(basq_ctx* ctx, RecPool* pool, int64_t off_glob, int S, const double* omega, const int* rank_excl,
                int K, bool scale_wf, int64_t dest_base, int64_t new_count);
int extract_result(basq_ctx* ctx, const RecPool& pool, int64_t idx_base, int64_t* idx_out, double* w_out);

// setsum.cu
struct SetSumArgs {
  const RecPool* pool;
  LmView lm;
  int64_t off_glob;   // global position of local record 0
  int S;              // set stride (number of sets)
  int64_t p_lo, p_hi; // local record range processed by this launch
  int nl;             // NlMode
  const double* corrT;  // [p_hi - p_lo, ld_corr] (non-linear modes) : A_z k(Xobs, x_p) per landmark
  int64_t ld_corr;
  const double* sz;     // per-landmark factor (non-linear modes)
  double* G;            // [lm->count, ldg]
  int64_t ldg;
  bool accumulate;
  double grid_m = 0.0;  // != 0: reproducible instances, terms rounded to the grid of 1.5 * 2^52 * Q (grid_round)
  double grid_m2 = 0.0; // fp64 records in reproducible instances: grid of the remainders term - hi, summed into G2
  double* G2 = nullptr; // [lm->count, ldg]
};
int set_sums(basq_ctx* ctx, const KParams& kp, const SetSumArgs& a);

// nlsum.cu: tensor-core set sums of the pairwise non-linear kernels (fp32 records)
struct NlOperands {
  int M = 0, n_obs = 0, KP = 0, n_mtiles = 0;
  float kx_scale = 1.f;
  DevBuf azh, azl, ainv, szf;   // Az = K(Z, Xobs) W as scaled fp16 hi / lo tiles, 1 / scale per row, fp32 landmark factors
  DevBuf kxh, kxl, trec;        // chunk buffers: k(Xobs, x) operand tiles and the tiles' candidate records
  size_t cap_tiles = 0, cap_rec_bytes = 0;
};
int nls_prepare(basq_ctx* ctx, const KParams& kp, const double* Az, int M, int n_obs, const double* sz,
                NlOperands* op);
int nls_set_sums(basq_ctx* ctx, const KParams& kp, int nl, NlOperands* op, const RecPool& pool, const LmView& lmz,
                 const LmView& lmobs, int64_t off, int S, int64_t p_lo, int64_t p_hi, double* G, int64_t ldg,
                 double grid_m = 0.0);

// gpvar.cu: fused posterior variance on the tensor cores (fp32 inputs)
// mean_out != NULL: the fused kernel also writes the posterior mean (*mean_done tells whether it did)
// At most GPV_MAX_OBS observations: KP^2 (the L^-1 operand tiles) stays inside int32 element indexing and the
// fp64 factor (8 n_obs^2 B) inside a few GB.  The variance kernels themselves do not depend on it.
constexpr int GPV_MAX_OBS = 32768;
int gp_variance_tc(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const LmView& lmobs, const void* X,
                   int64_t N, double* var_out, double* mean_out = nullptr, bool* mean_done = nullptr);

// dgemm.cu
int dgemm(basq_ctx* ctx, bool ta, bool tb, int m, int n, int k, double alpha, const double* A, int64_t lda,
          const double* B, int64_t ldb, double beta, double* C, int64_t ldc, bool b_lower_tri = false,
          bool a_lower_tri = false, bool c_symmetric = false, bool c_lower_only = false, bool fixed_order = false);
// fixed_order: one tile shape, no split-K - an element's k-sum does not depend on m or n (reproducible sessions)
// b_lower_tri (with tb): B is lower triangular, C = A B^T only visits k <= column
// a_lower_tri (without ta): A is lower triangular, C = A B only visits k <= row
// c_symmetric (m == n, beta == 0; e.g. A^T A): only the tiles that touch the lower triangle are computed, the
//   K range is split so that they still fill the SMs, and the upper triangle is the mirror image
// c_lower_only (m == n, any beta; e.g. the trailing update of a Cholesky factorisation): only the tiles that
//   touch the lower triangle are computed and written, nothing is mirrored; entries above the diagonal inside
//   those tiles are written too, the others keep their values

// car.cu
int caratheodory(basq_ctx* ctx, double* A, int n, int S, int lda, double* omega_out);

// api.cu: kernel(X, Y) [a, b] in fp64 (the body of basq_gram)
// diag_col0: X is rows [diag_col0, diag_col0 + a) of the square matrix kernel(Y, Y) - the diagonal terms
// (noise, jitter) then sit at (i, diag_col0 + i)
int gram_matrix(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t a, const void* Y, int64_t b,
                double* out, bool tensor_correction, int64_t diag_col0 = 0);
// The arrays a call evaluates the kernel on, in the precision it evaluates it in (sessions, weighted double sums).
// begin: fp64 inputs are narrowed to fp32 when the caller opted in (basq_ctx_allow_f32_eval; counts a demotion),
// Xobs_f64 then keeps the caller's observations.  promote: after the caller's conditioning guard tripped on an fp32
// evaluation, the call restarts in fp64 - on the caller's own arrays after a demotion, else on widened copies with
// the observations from Xobs_f64 (widened when it is NULL); counts a promotion.  After it can_promote is false.
struct EvalRoute {
  basq_kernel_desc desc;                   // what evaluation sees: dtype, Xobs
  const void* pts[2] = {nullptr, nullptr}; // the two point sets in desc.dtype (session: X, Z; double sums: X, Y)
  // b == a with nb == na (the symmetric double sum) shares one copy; a set of zero rows gets no copy
  int begin(basq_ctx* ctx, const basq_kernel_desc* caller, const void* a, int64_t na, const void* b, int64_t nb);
  bool can_promote(const basq_ctx* ctx) const { return desc.dtype == BASQ_F32 && ctx->kappa_max > 0.0; }
  int promote(basq_ctx* ctx);

 private:
  int copy_points(basq_ctx* ctx, int dtype);
  basq_kernel_desc caller_;
  const void* src_[2] = {nullptr, nullptr};
  int64_t rows_[2] = {0, 0};
  DevBuf copies_[3];   // the point sets and the observations in the other precision
  bool demoted_ = false;
};
// Landmark side of the posterior modes, shared by sessions and the weighted double sums (quadform.cu):
// Az[M, n_obs] = K(Z, Xobs) W for the prepared landmarks lmz (M = lmz.count) and the conditioning guard's
// kappa = max_m |Az_m|_1 (also stored in ctx->last_kappa; synchronises)
int posterior_az(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const LmView& lmz, double* Az,
                 double* kappa);
// set sums of the pairwise non-linear modes (WSABI-M, MMLT) against landmarks with Az and factors sz
struct NlSweep {
  int M = 0;
  bool use_nls = false;   // fp32 records: tensor-core operands (nlsum.cuh); else the chunked fp64-GEMM correction
  NlOperands nlop;
  const double* Az = nullptr;   // chunked path: the caller's Az, alive while sweeping
  DevBuf V, corrT;              // chunked path: k(Xobs, x) and the correction of a chunk of points
  int64_t chunkP = 0;
};
int nl_sweep_prepare(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const double* Az, int M,
                     const double* sz, int64_t N_loc, NlSweep* w);
// G[:, 0..S) for local records [p_lo, p_hi); a carries pool, landmarks, offset, S, nl, sz, G, ldg
int nl_sweep_sums(basq_ctx* ctx, const KParams& kp, int nl, NlSweep* w, const RecPool& pool, const LmView& lmz,
                  const LmView& lmobs, int64_t off, int S, int64_t p_lo, int64_t p_hi, double* G, int64_t ldg,
                  SetSumArgs* a);

// nystrom.cu
// out[rows, cols] fp64 N(0, 1) draws of the Philox stream `seed` (candidates.cu)
int standard_normals(basq_ctx* ctx, uint64_t seed, int64_t offset, int64_t rows, int cols, double* out);
// The ranks of a row-sharded Nystrom basis and the caller's exchange (basq_nystrom_basis_sharded)
struct NysShard {
  int rank = 0, world = 1;
  basq_exchange_fn fn = nullptr;
  void* user = nullptr;
  double* gram_buf = nullptr;   // [q, q], the buffer the exchange function all-reduces
  double* rows_buf = nullptr;   // [world * chunk, q], the buffer it all-gathers
};
// U_out [q, M]; shard == nullptr: this process holds all M rows.  S_out (Rayleigh quotients, may be NULL) only then.
int nystrom_basis(basq_ctx* ctx, const basq_kernel_desc* desc, const void* Z, int64_t M, int q,
                  const double* Omega, int niter, double* U_out, double* S_out, const NysShard* shard);

}  // namespace basq
