// C ABI of basq_b200 (include/basq_b200.h): context, kernel evaluations, staged recombination
// session and the single-call recombination loop.
#include <math.h>
#include <string.h>
#include <stdlib.h>

#include <algorithm>
#include <memory>
#include <new>

#include "common.cuh"
#include "igemm.cuh"
#include "tgemm.cuh"

namespace basq {
const char* last_error_cstr();

namespace {

__global__ void scale_columns_kernel(double* __restrict__ U, int rows, int cols, int64_t ld,
                                     const double* __restrict__ s) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)rows * cols) return;
  const int r = (int)(t / cols), c = (int)(t % cols);
  U[(int64_t)r * ld + c] *= s[c];
}

// out = f(C, fx, fy) elementwise for the warped kernels.  On the leading diagonal the likelihood
// noise enters the covariance BEFORE the warping (predictive_covariance adds it, BASQ/_gp.py:275-276,
// and wsabi*_kernel warp its result, BASQ/_wsabi.py:216-224), the jitter after it.
__global__ void warp_gram_kernel(double* __restrict__ C, int64_t a, int64_t b, int mode, const double* __restrict__ fx,
                                 const double* __restrict__ fy, double pre_add, double diag_add, int64_t diag_col0) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a * b) return;
  const int64_t i = t / b, j = t % b - diag_col0;   // row i of this block is row diag_col0 + i of the square matrix
  double c = C[t];
  if (i == j) c += pre_add;
  if (mode == BASQ_WSABI_L) c = fx[i] * c * fy[j + diag_col0];
  else if (mode == BASQ_WSABI_M) c = fx[i] * c * fy[j + diag_col0] + 0.5 * c * c;
  else if (mode == BASQ_MMLT_G) c = fx[i] * fy[j + diag_col0] * expm1(c);
  if (i == j) c += diag_add;
  C[t] = c;
}

// model-space moments of the warped GPs: wsabil_predict / wsabim_predict (BASQ/_wsabi.py:251-277),
// gspace_predict (SOBER/BASQ/_scale_mmlt.py:211-223)
__global__ void model_space_kernel(int mode, double offset, int64_t n, double* __restrict__ mean,
                                   double* __restrict__ var, int write_var) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const double m = mean[p];
  const double v = var ? var[p] : 0.0;
  double mo = m, vo = v;
  if (mode == BASQ_WSABI_L) { mo = offset + 0.5 * m * m; vo = m * v * m; }
  else if (mode == BASQ_WSABI_M) { mo = offset + 0.5 * (m * m + v); vo = m * v * m + 0.5 * v * v; }
  else if (mode == BASQ_MMLT_G) { mo = expm1(m + 0.5 * v); vo = mo * mo * expm1(v); }
  mean[p] = mo;
  if (write_var) var[p] = vo;
}

// out[m, i] = sum_{k < cnt} G[m, node[i] + k * stride]: the set-sum column of a tree node of the
// pass's cell hierarchy (a node = every stride-th cell from node[i]) in a fixed summation order
__global__ void fold_cols_kernel(const double* __restrict__ G, int64_t ldg, int rows, int K,
                                 const int* __restrict__ node, int stride, int cnt, double* __restrict__ out,
                                 int64_t ldo) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)rows * K) return;
  const int m = (int)(t / K), i = (int)(t % K);
  const double* src = G + (int64_t)m * ldg + node[i];
  double s = 0.0;
  for (int k = 0; k < cnt; ++k) s += src[(int64_t)k * stride];
  out[(int64_t)m * ldo + i] = s;
}

// raw[:, 0..K) holds the projected columns of the K nodes just folded.  Below level 0 they are the
// LOW halves of the K surviving parents and the HIGH halves follow by linearity,
// hi = parent - lo (parent = column ppos[i] of the previous level), so only half of a level's columns
// are ever projected.  A_out = columns scaled by the parents' factors fpar.
__global__ void level_finish_kernel(double* __restrict__ raw, const double* __restrict__ prev, int n, int K,
                                    int below0, const int* __restrict__ ppos, const double* __restrict__ fpar,
                                    double* __restrict__ A_out, int64_t ld) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)n * K) return;
  const int r = (int)(t / K), i = (int)(t % K);
  const double f = fpar[i];
  const double lo = raw[(int64_t)r * ld + i];
  A_out[(int64_t)r * ld + i] = f * lo;
  if (below0) {
    const double hi = prev[(int64_t)r * ld + ppos[i]] - lo;
    raw[(int64_t)r * ld + K + i] = hi;
    A_out[(int64_t)r * ld + K + i] = f * hi;
  }
}

__global__ void f32_to_f64_kernel(const float* __restrict__ in, int64_t n, double* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = (double)in[t];
}

__global__ void f64_to_f32_kernel(const double* __restrict__ in, int64_t n, float* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = (float)in[t];
}

// kappa = max over rows m of sum_o |A[m, o]|  (non-negative doubles order like their bit patterns)
__global__ void row_l1_max_kernel(const double* __restrict__ A, int rows, int cols, unsigned long long* __restrict__ out) {
  __shared__ double sh[256];
  const int m = blockIdx.x;
  double acc = 0.0;
  for (int o = threadIdx.x; o < cols; o += blockDim.x) acc += fabs(A[(int64_t)m * cols + o]);
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) atomicMax(out, (unsigned long long)__double_as_longlong(sh[0]));
}

// dst = src [rows, d] in `dtype`, converted from the other precision; zero rows get a one-row allocation
int convert_rows(basq_ctx* ctx, int dtype, const void* src, int64_t rows, int d, DevBuf* dst) {
  const size_t esz = dtype == BASQ_F32 ? sizeof(float) : sizeof(double);
  BASQ_TRY(dst->alloc(ctx, esz * (size_t)std::max<int64_t>(rows, 1) * d));
  const int64_t n = rows * d;
  if (n == 0) return BASQ_OK;
  if (dtype == BASQ_F32)
    f64_to_f32_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>((const double*)src, n, dst->as<float>());
  else
    f32_to_f64_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>((const float*)src, n, dst->as<double>());
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

}  // namespace

int EvalRoute::copy_points(basq_ctx* ctx, int dtype) {
  for (int i = 0; i < 2; ++i) {
    if (i == 1 && src_[1] == src_[0] && rows_[1] == rows_[0]) {
      pts[1] = pts[0];
      break;
    }
    BASQ_TRY(convert_rows(ctx, dtype, src_[i], rows_[i], caller_.d, &copies_[i]));
    pts[i] = copies_[i].p;
  }
  return BASQ_OK;
}

int EvalRoute::begin(basq_ctx* ctx, const basq_kernel_desc* caller, const void* a, int64_t na, const void* b,
                     int64_t nb) {
  desc = caller_ = *caller;
  pts[0] = src_[0] = a;
  pts[1] = src_[1] = b;
  rows_[0] = na;
  rows_[1] = nb;
  if (caller->dtype != BASQ_F64 || !ctx->eval_f32) return BASQ_OK;
  // opt-in: evaluate the kernel in fp32 (tensor-core set sums) although the caller's arrays are fp64 - SOBER runs
  // everything in torch.double (SOBER/_settings.py:4-11); accumulation, projection and Caratheodory stay fp64 as on
  // the fp32 path, and the caller's conditioning guard may still send the call back to fp64
  BASQ_TRY(copy_points(ctx, BASQ_F32));
  if (caller->mode != BASQ_PLAIN) {
    BASQ_TRY(convert_rows(ctx, BASQ_F32, caller->Xobs, caller->n_obs, caller->d, &copies_[2]));
    desc.Xobs = copies_[2].p;
    desc.Xobs_f64 = static_cast<const double*>(caller->Xobs);
  }
  desc.dtype = BASQ_F32;
  demoted_ = true;
  ctx->demotions++;
  return BASQ_OK;
}

int EvalRoute::promote(basq_ctx* ctx) {
  ctx->promotions++;
  if (demoted_) {   // the caller's arrays were fp64 to begin with: go back to them
    for (DevBuf& c : copies_) c.release();
    desc = caller_;
    pts[0] = src_[0];
    pts[1] = src_[1];
    return BASQ_OK;
  }
  BASQ_TRY(copy_points(ctx, BASQ_F64));
  if (desc.mode != BASQ_PLAIN) {
    if (desc.Xobs_f64) {
      desc.Xobs = desc.Xobs_f64;   // W belongs to these coordinates, not to their fp32 roundings
    } else {
      BASQ_TRY(convert_rows(ctx, BASQ_F64, desc.Xobs, desc.n_obs, desc.d, &copies_[2]));
      desc.Xobs = copies_[2].p;
    }
  }
  desc.dtype = BASQ_F64;
  return BASQ_OK;
}

namespace {

int check_finite_host(const double* v, int64_t n, const char* what) {
  for (int64_t i = 0; i < n; ++i)
    BASQ_CHECK(isfinite(v[i]), BASQ_ERR_NUMERIC, "%s contains a non-finite value at %lld", what, (long long)i);
  return BASQ_OK;
}

}  // namespace
}  // namespace basq

using namespace basq;

// =============================================================================================
// session
// =============================================================================================
struct Piece {   // a typed view of a slice of the context's host-call buffer (basq_recombine_host)
  void* p = nullptr;
  template <typename T> T* as() const { return static_cast<T*>(p); }
};

// Sessions with at least this many basis rows q and landmark rows Mtot project their level columns on the int8
// tensor cores (scripts/time_projection.py, B200 at 1000 W: GEMM kernel 2.7-3.3x faster than the fp64 GEMM at
// q = 999, Mtot = 10000-11002); below, slicing the level columns eats the gain (q = 499, Mtot = 5000: 0.15 ms
// kernel + 0.05 ms slicing against 0.24 ms) and the fp64 GEMM stays.
constexpr int INT8_PROJ_MIN_Q = 512, INT8_PROJ_MIN_MTOT = 8192;

struct basq_session {
  basq_ctx* ctx = nullptr;
  basq_kernel_desc desc;
  KParams kp;
  int M = 0, q = 0, n = 0, S = 0, Mtot = 0;
  int nl = NL_LIN;
  Landmarks lm;     // Z (+ Xobs appended for the linear posterior-covariance modes)
  Landmarks lmobs;  // Xobs alone
  DevBuf Uprime;    // [q, Mtot]
  // Large sessions project on the int8 tensor cores (igemm.cu): U' as digits once, the level columns per level.
  // Decided once per session: hi = parent - lo mixes the projections of two levels, which must share one arithmetic.
  bool int8_proj = false;
  DigOperand Udig, Gdig;
  DevBuf sz;        // [M] per-landmark factor
  DevBuf Az;        // [M, n_obs] = K(Z, Xobs) W          (non-linear modes)
  RecPool pool;
  DevBuf G;         // [Mtot, ldg]   (ldg = cells of the widest pass so far)
  int64_t ldg = 0;
  DevBuf rank;      // int [cells]
  // state of the current pass (session_pass_begin / session_level)
  int pass_F = 0;
  int64_t pass_R = 0, pass_off = 0;
  const double* obj = nullptr;  // [N_loc] objective per original local row (objective-aware mode), or NULL
  int rows = 0;                 // rows of a level system: n, or n + 1 with the objective row
  DevBuf cellmass;  // [cells] mass of every cell
  DevBuf cellobj;   // [cells] objective sum of every cell
  DevBuf Gf;        // [Mtot, S] folded set-sum columns of a level
  DevBuf raw[2];    // [n, S] unscaled local columns of the current / previous level
  int raw_cur = 0;
  DevBuf lnode, lppos, lfpar;  // device copies of a level's node ids, parent positions, parent factors
  NlSweep nls;      // set sums of the non-linear modes (tensor-core operands or chunk buffers)
  // the precision the session evaluates in (session_create_impl); holds the narrowed or widened input copies
  EvalRoute route;
  double kappa = 0.0;
  int64_t idx_base = 0;
  bool scale_wf = true;
  // reproducible mode (basq_ctx_reproducible at creation): the next pass sums on the grids set by
  // session_set_grid for grid_R live points - set sums, masses, objective (1.5 * 2^52 * Q each, grid_round)
  bool repro = false;
  double szmax = 0.0;   // max_m |sz_m| (non-linear modes): enters the bound of the set sums
  int64_t grid_R = -1;
  double grid_m[3] = {0.0, 0.0, 0.0};
  double grid_m2[3] = {0.0, 0.0, 0.0};  // the finer grids of the remainders of fp64 terms (hi / lo, set_grid)
  DevBuf G2, cellmass2, cellobj2;      // the sums of those remainders (G2: fp64 records only)
  DevBuf Gc;                           // [Mtot + 2, S] hi + lo of the summed exact columns (project_exact)
  std::vector<double> omega_host;
  std::vector<int> rank_host;
};

namespace basq {
namespace {

// G[:, 0..ncols) for local records [p_lo, p_hi), set index = (off + p) mod S; grid_m != 0: on that grid
int session_set_sums(basq_session* s, int64_t off, int S, int64_t p_lo, int64_t p_hi, double* G, int64_t ldg,
                     double grid_m = 0.0, double grid_m2 = 0.0, double* G2 = nullptr) {
  basq_ctx* ctx = s->ctx;
  SetSumArgs a;
  a.grid_m = grid_m;
  a.grid_m2 = grid_m2;
  a.G2 = G2;
  a.pool = &s->pool;
  a.lm = s->lm.view();
  a.off_glob = off;
  a.S = S;
  a.nl = s->nl;
  a.sz = s->sz.as<double>();
  a.G = G;
  a.ldg = ldg;
  if (s->nl == NL_LIN) {
    a.p_lo = p_lo;
    a.p_hi = p_hi;
    a.corrT = nullptr;
    a.ld_corr = 0;
    a.accumulate = false;
    return set_sums(ctx, s->kp, a);
  }
  return nl_sweep_sums(ctx, s->kp, s->nl, &s->nls, s->pool, s->lm.view(), s->lmobs.view(), off, S, p_lo, p_hi, G, ldg,
                       &a);
}

}  // namespace

// Az = K(Z, Xobs) W   (BASQ/_gp.py:270-273: KxX @ woodbury_inv) and the conditioning guard's measure.  The
// correction K_ZX W k(Xobs, x) multiplies the kernel values by the rows of Az, so an evaluation error eps_k of
// k (fp32: ~2e-7 relative) reaches the covariance as eps_k |Az_m|_1 sigma_f^2.  kappa = max_m |Az_m|_1 is
// O(10) for well-separated observations even at the reference's default noise 1e-10 (BASQ/_parameters.py:30),
// but grows like sigma_f / sigma_n for clustered ones; beyond kappa_max the fp32 inputs are promoted to the
// all-fp64 path.
int posterior_az(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const LmView& lmz, double* Az,
                 double* kappa) {
  const int M = lmz.count, n_obs = desc->n_obs;
  DevBuf KzX, kap;
  BASQ_TRY(KzX.alloc(ctx, sizeof(double) * (size_t)M * n_obs));
  BASQ_TRY(base_gram(ctx, kp, lmz, desc->Xobs, n_obs, KzX.as<double>(), n_obs));
  BASQ_TRY(dgemm(ctx, false, false, M, n_obs, n_obs, 1.0, KzX.as<double>(), n_obs, desc->W, n_obs, 0.0, Az, n_obs));
  BASQ_TRY(kap.alloc(ctx, sizeof(unsigned long long)));
  BASQ_CUDA(cudaMemsetAsync(kap.p, 0, sizeof(unsigned long long), ctx->stream));
  row_l1_max_kernel<<<(unsigned)M, 256, 0, ctx->stream>>>(Az, M, n_obs, kap.as<unsigned long long>());
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  BASQ_CUDA(cudaMemcpyAsync(kappa, kap.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));  // also: KzX goes out of scope
  BASQ_CHECK(isfinite(*kappa), BASQ_ERR_NUMERIC, "the GP caches contain non-finite values (K_ZX W)");
  ctx->last_kappa = *kappa;
  return BASQ_OK;
}

// Non-linear modes: fp32 records run on the tensor cores (nlsum.cuh, operands from Az); otherwise the
// correction is built per chunk of points, whose size is chosen here for N_loc points.  Az stays the caller's
// and must outlive the sweeps on the chunked path.
int nl_sweep_prepare(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const double* Az, int M,
                     const double* sz, int64_t N_loc, NlSweep* w) {
  const int n_obs = desc->n_obs;
  { const char* t = getenv("BASQ_NLSUM"); ctx->no_nlsum = t && t[0] == '0'; }  // read per call (A/B tests toggle it)
  w->M = M;
  w->Az = Az;
  w->use_nls = desc->dtype == BASQ_F32 && !ctx->no_nlsum;
  if (w->use_nls) {
    // fp32 records: the pairwise correction runs on the tensor cores (nlsum.cuh)
    BASQ_TRY(nls_prepare(ctx, kp, Az, M, n_obs, sz, &w->nlop));
    w->Az = nullptr;
  } else {
    // points per chunk of the pairwise correction: corrT [P, M] may take up to 2 GB, so that a chunk
    // spans many cells of a refined pass (every chunk re-reads the G columns it touches)
    int64_t P = (int64_t)(2048ll << 20) / (8ll * std::max<int64_t>(M, n_obs));
    P = std::max<int64_t>(1024, std::min<int64_t>(P, 131072));
    P = std::min<int64_t>(P, std::max<int64_t>(N_loc, 1024));
    w->chunkP = P;
    BASQ_TRY(w->V.alloc(ctx, sizeof(double) * (size_t)n_obs * P));
    BASQ_TRY(w->corrT.alloc(ctx, sizeof(double) * (size_t)M * P));
  }
  return BASQ_OK;
}

// G[:, 0..S) of the non-linear set sums of local records [p_lo, p_hi); a = the set-sum arguments of the linear
// fields (pool, landmarks, offset, sets, G, sz), completed here per chunk.
int nl_sweep_sums(basq_ctx* ctx, const KParams& kp, int nl, NlSweep* w, const RecPool& pool, const LmView& lmz,
                  const LmView& lmobs, int64_t off, int S, int64_t p_lo, int64_t p_hi, double* G, int64_t ldg,
                  SetSumArgs* a) {
  if (w->use_nls) return nls_set_sums(ctx, kp, nl, &w->nlop, pool, lmz, lmobs, off, S, p_lo, p_hi, G, ldg, a->grid_m);
  // non-linear kernels need C_h(z_m, x_p) = k(z_m, x_p) - (K_ZX W) k(Xobs, x_p) per pair: build the
  // correction for a chunk of points with two GEMM-shaped steps, then accumulate.
  const int n_obs = lmobs.count;
  BASQ_CUDA(cudaMemsetAsync(G, 0, sizeof(double) * (size_t)lmz.count * ldg, ctx->stream));
  if (a->G2) BASQ_CUDA(cudaMemsetAsync(a->G2, 0, sizeof(double) * (size_t)lmz.count * ldg, ctx->stream));
  for (int64_t c0 = p_lo; c0 < p_hi; c0 += w->chunkP) {
    const int64_t c1 = std::min(p_hi, c0 + w->chunkP);
    const int64_t cnt = c1 - c0;
    BASQ_TRY(base_gram_records(ctx, kp, lmobs, pool, c0, c1, w->V.as<double>(), w->chunkP));
    // corrT[p, m] = sum_o V[o, p] * Az[m, o]; in reproducible sessions a point's correction must not depend on
    // the chunk it falls into (the chunk sizes depend on the shard), so the GEMM runs in a fixed summation order
    BASQ_TRY(dgemm(ctx, true, true, (int)cnt, w->M, n_obs, 1.0, w->V.as<double>(), w->chunkP, w->Az, n_obs, 0.0,
                   w->corrT.as<double>(), w->M, false, false, false, false, a->grid_m != 0.0));
    a->p_lo = c0;
    a->p_hi = c1;
    a->corrT = w->corrT.as<double>();
    a->ld_corr = w->M;
    a->accumulate = true;
    BASQ_TRY(set_sums(ctx, kp, *a));
  }
  return BASQ_OK;
}

namespace {

int session_create_impl(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N_loc, int64_t N_glob,
                        int64_t idx_base, const void* Z, int64_t M, const double* U, int q, const double* mu,
                        int S_override, basq_session* s) {
  PhaseTimer timer(ctx, PH_PREP);
  BASQ_CHECK(ctx && desc && Z && U, BASQ_ERR_INVALID, "session: NULL argument");
  BASQ_CHECK(N_loc >= 0 && (X || N_loc == 0), BASQ_ERR_INVALID, "session: bad candidate buffer");
  BASQ_CHECK(q >= 1 && M >= q, BASQ_ERR_INVALID, "session: need 1 <= q <= M (q=%d, M=%lld)", q, (long long)M);
  BASQ_CHECK(M <= 1000000, BASQ_ERR_UNSUPPORTED, "session: more than 1e6 landmarks");
  s->ctx = ctx;
  s->M = (int)M;
  s->q = q;
  s->n = q + 1;
  s->rows = s->n;
  s->S = S_override > 0 ? S_override : 2 * (q + 1);
  s->idx_base = idx_base;
  s->repro = ctx->reproducible;
  const int mode = desc->mode;
  const int n_obs = (mode == BASQ_PLAIN) ? 0 : desc->n_obs;
  const bool nonlin = (mode == BASQ_WSABI_M || mode == BASQ_MMLT_G);
  s->nl = mode == BASQ_WSABI_M ? NL_WSABIM : (mode == BASQ_MMLT_G ? NL_MMLT : NL_LIN);
  s->scale_wf = !nonlin;
  const bool augment = (mode == BASQ_PRED_COV || mode == BASQ_WSABI_L);

  // From here on the session evaluates on the route's arrays.  At most two attempts: an fp32 one whose conditioning
  // guard trips is dropped and redone in fp64.
  BASQ_TRY(s->route.begin(ctx, desc, X, N_loc, Z, M));
  for (;;) {
    desc = &s->route.desc;
    X = s->route.pts[0];
    Z = s->route.pts[1];
    s->desc = *desc;
    BASQ_TRY(make_kparams(desc, &s->kp));
    BASQ_TRY(compute_center(ctx, desc, Z, M, &s->kp));
    if (mode != BASQ_PLAIN) BASQ_TRY(prep_landmarks(ctx, s->kp, desc->dtype, desc->Xobs, n_obs, nullptr, 0, &s->lmobs));
    BASQ_TRY(prep_landmarks(ctx, s->kp, desc->dtype, Z, M, augment ? desc->Xobs : nullptr, augment ? n_obs : 0, &s->lm));
    s->Mtot = s->lm.count;
    if (mode == BASQ_PLAIN) break;
    BASQ_TRY(s->Az.alloc(ctx, sizeof(double) * (size_t)M * n_obs));
    BASQ_TRY(posterior_az(ctx, desc, s->kp, s->lm.view(0, (int)M), s->Az.as<double>(), &s->kappa));
    if (!(s->route.can_promote(ctx) && s->kappa > ctx->kappa_max)) break;
    s->lm.release();
    s->lmobs.release();
    s->Az.release();
    BASQ_TRY(s->route.promote(ctx));
  }

  // per-landmark and per-point factors of the warped kernels
  DevBuf sx;
  const bool has_factor = (mode == BASQ_WSABI_L || mode == BASQ_WSABI_M || mode == BASQ_MMLT_G);
  if (has_factor) {
    BASQ_TRY(s->sz.alloc(ctx, sizeof(double) * M));
    BASQ_TRY(warp_factor(ctx, desc, s->kp, s->lmobs.view(), Z, M, s->sz.as<double>()));
    BASQ_TRY(sx.alloc(ctx, sizeof(double) * std::max<int64_t>(N_loc, 1)));
    BASQ_TRY(warp_factor(ctx, desc, s->kp, s->lmobs.view(), X, N_loc, sx.as<double>()));
    if (s->repro && nonlin) {   // replicated landmark data: the same maximum on every rank
      std::vector<double> h((size_t)M);
      BASQ_CUDA(cudaMemcpyAsync(h.data(), s->sz.p, sizeof(double) * M, cudaMemcpyDeviceToHost, ctx->stream));
      BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
      for (double v : h) s->szmax = std::max(s->szmax, fabs(v));
      BASQ_CHECK(isfinite(s->szmax), BASQ_ERR_NUMERIC, "session: non-finite warp factor of a landmark");
    }
  }

  // projection matrix U' [q, Mtot]
  BASQ_TRY(s->Uprime.alloc(ctx, sizeof(double) * (size_t)q * s->Mtot));
  BASQ_CUDA(cudaMemcpy2DAsync(s->Uprime.p, sizeof(double) * s->Mtot, U, sizeof(double) * M, sizeof(double) * M, q,
                              cudaMemcpyDeviceToDevice, ctx->stream));
  if (mode == BASQ_WSABI_L) {
    scale_columns_kernel<<<ceil_div((int64_t)q * M, 256), 256, 0, ctx->stream>>>(s->Uprime.as<double>(), q, (int)M,
                                                                                s->Mtot, s->sz.as<double>());
    ctx->launches++;
  }
  if (augment) {
    // U'[:, M:] = -(U diag(sz)) Az : the posterior-covariance correction folded into the projection
    BASQ_TRY(dgemm(ctx, false, false, q, n_obs, (int)M, -1.0, s->Uprime.as<double>(), s->Mtot, s->Az.as<double>(),
                   n_obs, 0.0, s->Uprime.as<double>() + M, s->Mtot));
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
    s->Az.release();
  }
  s->int8_proj = q >= INT8_PROJ_MIN_Q && s->Mtot >= INT8_PROJ_MIN_MTOT;
  if (s->int8_proj) BASQ_TRY(dig_from_f64(ctx, s->Uprime.as<double>(), s->Mtot, false, q, s->Mtot, 0, 128, &s->Udig));

  // candidate records
  const double uniform_w = 1.0 / (double)(N_glob > 0 ? N_glob : 1);
  BASQ_TRY(build_records(ctx, s->kp, desc->dtype, X, N_loc, uniform_w, mu, has_factor ? sx.as<double>() : nullptr,
                         !nonlin, &s->pool));

  s->ldg = 0;  // G and the rank table are sized by the first pass (session_reserve_cells)
  if (nonlin) {
    BASQ_TRY(nl_sweep_prepare(ctx, desc, s->kp, s->Az.as<double>(), (int)M, s->sz.as<double>(), N_loc, &s->nls));
    if (s->nls.use_nls) s->Az.release();
  }
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));  // sx goes out of scope
  return BASQ_OK;
}

// buffers that scale with the number of cells (F * S) of a pass
int session_reserve_cells(basq_session* s, int cells) {
  if (cells <= s->ldg) return BASQ_OK;
  basq_ctx* ctx = s->ctx;
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  s->G.release();
  s->rank.release();
  s->ldg = cells;
  BASQ_TRY(s->G.alloc(ctx, sizeof(double) * (size_t)s->Mtot * s->ldg));
  BASQ_TRY(s->rank.alloc(ctx, sizeof(int) * (size_t)cells));
  s->cellmass.release();
  s->cellobj.release();
  BASQ_TRY(s->cellmass.alloc(ctx, sizeof(double) * (size_t)cells));
  BASQ_TRY(s->cellobj.alloc(ctx, sizeof(double) * (size_t)cells));
  if (s->repro) {
    s->G2.release();
    s->cellmass2.release();
    s->cellobj2.release();
    if (s->pool.dtype == BASQ_F64) BASQ_TRY(s->G2.alloc(ctx, sizeof(double) * (size_t)s->Mtot * s->ldg));
    BASQ_TRY(s->cellmass2.alloc(ctx, sizeof(double) * (size_t)cells));
    BASQ_TRY(s->cellobj2.alloc(ctx, sizeof(double) * (size_t)cells));
  }
  s->omega_host.resize(cells);
  s->rank_host.resize(cells);
  return BASQ_OK;
}

// Begin a pass over F * S cells (cell of a point = global position mod F * S; set j = cells j,
// j + S, ..., j + (F-1) S).  ONE sweep of kernel evaluations fills G[:, c] = sum over cell c of
// w_p k(z, x_p); the log2(F) + 1 Caratheodory levels of the pass (session_level) then only fold and
// project columns of G.  F = 1 is the reference's round (BASQ/_rchq.py:81-101).
int session_pass_begin(basq_session* s, int64_t R_glob, int64_t off, int F) {
  basq_ctx* ctx = s->ctx;
  BASQ_CHECK(F >= 1 && F <= BASQ_MAX_CELL_FACTOR && (F & (F - 1)) == 0, BASQ_ERR_INVALID,
             "pass: the cell factor must be a power of two <= %d (got %d)", BASQ_MAX_CELL_FACTOR, F);
  const int cells = F * s->S;
  BASQ_CHECK(F == 1 || R_glob >= cells, BASQ_ERR_INVALID, "pass: refined passes need R >= F * S");
  BASQ_CHECK(off >= 0 && off + s->pool.count <= R_glob, BASQ_ERR_INVALID,
             "pass: offset %lld + local %lld exceeds global %lld", (long long)off, (long long)s->pool.count,
             (long long)R_glob);
  BASQ_CHECK(!s->repro || s->grid_R == R_glob, BASQ_ERR_INVALID,
             "pass: a reproducible session needs the grids of this pass first (basq_session_set_grid)");
  const int c_eff = (int)std::min<int64_t>(cells, R_glob);
  BASQ_TRY(session_reserve_cells(s, cells));
  if (!s->Gf.p) {
    // reproducible sessions: hi and lo parts of the set sums, masses and objective sums (session_level_fold_exact)
    BASQ_TRY(s->Gf.alloc(ctx, sizeof(double) * (size_t)(s->repro ? 2 * (s->Mtot + 2) : s->Mtot) * s->S));
    if (s->repro) BASQ_TRY(s->Gc.alloc(ctx, sizeof(double) * (size_t)(s->Mtot + 2) * s->S));
    for (int i = 0; i < 2; ++i) BASQ_TRY(s->raw[i].alloc(ctx, sizeof(double) * (size_t)(s->n + 1) * s->S));
    BASQ_TRY(s->lnode.alloc(ctx, sizeof(int) * s->S));
    BASQ_TRY(s->lppos.alloc(ctx, sizeof(int) * s->S));
    BASQ_TRY(s->lfpar.alloc(ctx, sizeof(double) * s->S));
  }
  s->pass_F = F;
  s->pass_R = R_glob;
  s->pass_off = off;
  PhaseTimer t(ctx, PH_SETSUM);
  BASQ_TRY(set_masses(ctx, s->pool, off, cells, c_eff, s->cellmass.as<double>(), s->grid_m[1], s->grid_m2[1],
                      s->cellmass2.as<double>()));
  if (s->obj)
    BASQ_TRY(cell_objective(ctx, s->pool, off, cells, c_eff, s->obj, s->cellobj.as<double>(), s->grid_m[2],
                            s->grid_m2[2], s->cellobj2.as<double>()));
  BASQ_TRY(session_set_sums(s, off, cells, 0, s->pool.count, s->G.as<double>(), s->ldg, s->grid_m[0], s->grid_m2[0],
                            s->G2.as<double>()));
  s->grid_R = -1;   // the grids belong to this pass
  return BASQ_OK;
}

// Local part of level `lvl` of the current pass: A_out[n, S] (ld = S, columns beyond the level's
// count zero), row 0 = masses, rows 1..q = U' G (reference: U_svd @ X_for_nys, BASQ/_rchq.py:88).
//   lvl 0: K columns, column i = set node[i] (all F cells of it), scaled by fpar[i].
//   lvl > 0: 2 K columns [low halves | high halves] of the K surviving nodes of the previous level;
//            node[i] = id of the low half (cells node[i] + k (S << lvl)), ppos[i] = the parent's column
//            in the previous level, fpar[i] = the parent's factor; high half = parent - low half.
// The two halves of session_level, also exposed on their own so that ranks can exchange the folded
// columns between them (sharded.py: reduce-scatter by landmark rows, every rank then projects 1/G of
// the rows instead of all of them).
//   fold:    Gf_out[m, i] = sum_k G[m, node[i] + k (S << lvl)]   for m < Mtot, i < K   (ld = ld_gf)
//   project: rows 1..q of the level's raw columns = U'[:, row0 .. row0 + nrows) Gf_rows[nrows, K];
//            masses / objective rows from this rank's cells; high halves by linearity; A_out scaled.
// Pinned staging ring of the context for the small per-level host arrays (node ids, parent positions, parent
// factors): the H2D copies read from a slot of this ring, so the level calls return without synchronising the
// stream and the caller may reuse its arrays at once; a slot is reused only after the event recorded behind
// its copies.  Allocated once per context (cudaHostAlloc / cudaFreeHost synchronise the device).
int stage_take(basq_ctx* ctx, size_t bytes, unsigned char** slot_out, int* slot_index) {
  if (bytes > ctx->stage_slot_bytes) {
    if (ctx->stage) {
      BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
      BASQ_CUDA(cudaFreeHost(ctx->stage));
      ctx->stage = nullptr;
    }
    const size_t slot = std::max<size_t>(bytes, 64 << 10);
    BASQ_CUDA(cudaHostAlloc((void**)&ctx->stage, slot * basq_ctx::STAGE_SLOTS, cudaHostAllocDefault));
    ctx->stage_slot_bytes = slot;
    for (int i = 0; i < basq_ctx::STAGE_SLOTS; ++i)
      if (!ctx->stage_ev[i]) BASQ_CUDA(cudaEventCreateWithFlags(&ctx->stage_ev[i], cudaEventDisableTiming));
  }
  const int i = ctx->stage_next;
  ctx->stage_next = (ctx->stage_next + 1) % basq_ctx::STAGE_SLOTS;
  BASQ_CUDA(cudaEventSynchronize(ctx->stage_ev[i]));   // returns at once for a never-recorded / completed event
  *slot_out = ctx->stage + (size_t)i * ctx->stage_slot_bytes;
  *slot_index = i;
  return BASQ_OK;
}

int session_level_check(basq_session* s, int lvl, int K, const int* node_host, const int* ppos_host) {
  const int S = s->S, F = s->pass_F;
  BASQ_CHECK(F >= 1 && lvl >= 0 && (1 << lvl) <= F, BASQ_ERR_INVALID, "level %d outside the pass (F = %d)", lvl, F);
  const int C = lvl == 0 ? K : 2 * K;
  BASQ_CHECK(K >= 1 && C <= S, BASQ_ERR_INVALID, "level %d: %d columns exceed S = %d", lvl, C, S);
  const int stride = S << lvl;
  for (int i = 0; i < K; ++i)
    BASQ_CHECK(node_host[i] >= 0 && node_host[i] < stride &&
                   (lvl == 0 || !ppos_host || (ppos_host[i] >= 0 && ppos_host[i] < S)),
               BASQ_ERR_INVALID, "level %d: bad node %d", lvl, i);
  return BASQ_OK;
}

int session_level_fold(basq_session* s, int lvl, int K, const int* node_host, double* Gf_out, int64_t ld_gf) {
  basq_ctx* ctx = s->ctx;
  BASQ_TRY(session_level_check(s, lvl, K, node_host, nullptr));
  PhaseTimer t(ctx, PH_PROJ);
  const int stride = s->S << lvl, cnt = s->pass_F >> lvl;
  unsigned char* slot = nullptr;
  int si = 0;
  BASQ_TRY(stage_take(ctx, (size_t)s->S * 16, &slot, &si));
  memcpy(slot, node_host, sizeof(int) * K);
  BASQ_CUDA(cudaMemcpyAsync(s->lnode.p, slot, sizeof(int) * K, cudaMemcpyHostToDevice, ctx->stream));
  BASQ_CUDA(cudaEventRecord(ctx->stage_ev[si], ctx->stream));
  fold_cols_kernel<<<(unsigned)ceil_div64((int64_t)s->Mtot * K, 256), 256, 0, ctx->stream>>>(
      s->G.as<double>(), s->ldg, s->Mtot, K, s->lnode.as<int>(), stride, cnt, Gf_out, ld_gf);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;   // no synchronisation: node_host was copied into the pinned ring
}

// exact: Gf_rows holds all Mtot + 2 rows of session_level_fold_exact summed over the ranks; masses and
// objective sums come from its last two rows instead of this rank's cells
int session_level_project(basq_session* s, int lvl, int K, const int* node_host, const int* ppos_host,
                          const double* fpar_host, const double* Gf_rows, int64_t ld_gf, int row0, int nrows,
                          double* A_out, bool exact = false) {
  basq_ctx* ctx = s->ctx;
  const int n = s->n, S = s->S, F = s->pass_F, rows = s->rows;
  BASQ_TRY(session_level_check(s, lvl, K, node_host, ppos_host));
  BASQ_CHECK(row0 >= 0 && nrows >= 0 && row0 + nrows <= s->Mtot, BASQ_ERR_INVALID, "level: bad landmark row range");
  const int stride = S << lvl, cnt = F >> lvl;
  PhaseTimer t(ctx, PH_PROJ);
  {
    unsigned char* slot = nullptr;
    int si = 0;
    BASQ_TRY(stage_take(ctx, (size_t)s->S * 16, &slot, &si));
    int* h_node = reinterpret_cast<int*>(slot);
    int* h_ppos = h_node + S;
    double* h_fpar = reinterpret_cast<double*>(slot + (size_t)S * 8);
    memcpy(h_node, node_host, sizeof(int) * K);
    if (lvl > 0) memcpy(h_ppos, ppos_host, sizeof(int) * K);
    memcpy(h_fpar, fpar_host, sizeof(double) * K);
    BASQ_CUDA(cudaMemcpyAsync(s->lnode.p, h_node, sizeof(int) * K, cudaMemcpyHostToDevice, ctx->stream));
    if (lvl > 0) BASQ_CUDA(cudaMemcpyAsync(s->lppos.p, h_ppos, sizeof(int) * K, cudaMemcpyHostToDevice, ctx->stream));
    BASQ_CUDA(cudaMemcpyAsync(s->lfpar.p, h_fpar, sizeof(double) * K, cudaMemcpyHostToDevice, ctx->stream));
    BASQ_CUDA(cudaEventRecord(ctx->stage_ev[si], ctx->stream));
  }
  BASQ_CUDA(cudaMemsetAsync(A_out, 0, sizeof(double) * (size_t)rows * S, ctx->stream));
  double* raw = s->raw[s->raw_cur].as<double>();
  const double* prev = s->raw[s->raw_cur ^ 1].as<double>();
  if (exact) {
    BASQ_CUDA(cudaMemcpyAsync(raw, Gf_rows + (int64_t)s->Mtot * ld_gf, sizeof(double) * K, cudaMemcpyDeviceToDevice,
                              ctx->stream));
    if (s->obj)
      BASQ_CUDA(cudaMemcpyAsync(raw + (int64_t)n * S, Gf_rows + (int64_t)(s->Mtot + 1) * ld_gf, sizeof(double) * K,
                                cudaMemcpyDeviceToDevice, ctx->stream));
  } else {
    fold_cols_kernel<<<(unsigned)ceil_div64(K, 256), 256, 0, ctx->stream>>>(s->cellmass.as<double>(), 0, 1, K,
                                                                            s->lnode.as<int>(), stride, cnt, raw, S);
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
  }
  if (s->obj && !exact) {  // objective row (SOBER/_rchq.py:138-146), folded like the masses
    fold_cols_kernel<<<(unsigned)ceil_div64(K, 256), 256, 0, ctx->stream>>>(s->cellobj.as<double>(), 0, 1, K,
                                                                            s->lnode.as<int>(), stride, cnt,
                                                                            raw + (int64_t)n * S, S);
    ctx->launches++;
  }
  if (nrows > 0 && s->int8_proj) {
    BASQ_TRY(dig_from_f64(ctx, Gf_rows, ld_gf, true, K, nrows, row0, 64, &s->Gdig));
    BASQ_TRY(igemm(ctx, s->Udig, s->Gdig, 1.0, raw + S, S, false));
  } else if (nrows > 0) {
    BASQ_TRY(dgemm(ctx, false, false, s->q, K, nrows, 1.0, s->Uprime.as<double>() + row0, s->Mtot, Gf_rows, ld_gf, 0.0,
                   raw + S, S));
  } else {
    BASQ_CUDA(cudaMemset2DAsync(raw + S, sizeof(double) * S, 0, sizeof(double) * K, s->q, ctx->stream));
  }
  level_finish_kernel<<<(unsigned)ceil_div64((int64_t)rows * K, 256), 256, 0, ctx->stream>>>(
      raw, prev, rows, K, lvl > 0 ? 1 : 0, s->lppos.as<int>(), s->lfpar.as<double>(), A_out, S);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  // no synchronisation: the host arrays were copied into the pinned ring and may be reused at once
  s->raw_cur ^= 1;
  return BASQ_OK;
}

// Reproducible sessions: the level's grid-exact columns of this rank, Gf_out[2 (Mtot + 2), K] (ld = ld_gf): rows
// 0 .. Mtot-1 the folded set sums, row Mtot the masses, row Mtot + 1 the objective sums (0 without objective), on
// the pass's grids; rows Mtot + 2 .. 2 Mtot + 3 the same for the remainders on the finer grids (0 where a sum has
// one grid: set sums of fp32 records).  Every entry is a multiple of its grid and far from overflowing it, so the
// fold, and any sum of these arrays over ranks in any order, is exact.
int session_level_fold_exact(basq_session* s, int lvl, int K, const int* node_host, double* Gf_out, int64_t ld_gf) {
  basq_ctx* ctx = s->ctx;
  BASQ_CHECK(s->repro, BASQ_ERR_INVALID, "level_fold_exact: the session is not reproducible (basq_ctx_reproducible)");
  BASQ_TRY(session_level_fold(s, lvl, K, node_host, Gf_out, ld_gf));   // also copies node_host to s->lnode
  const int stride = s->S << lvl, cnt = s->pass_F >> lvl, Mtot = s->Mtot;
  double* lo = Gf_out + (int64_t)(Mtot + 2) * ld_gf;
  auto fold = [&](const DevBuf& src, int rows, int64_t ldsrc, double* dst) {
    fold_cols_kernel<<<(unsigned)ceil_div64((int64_t)rows * K, 256), 256, 0, ctx->stream>>>(
        src.as<double>(), ldsrc, rows, K, s->lnode.as<int>(), stride, cnt, dst, ld_gf);
    ctx->launches++;
  };
  auto zero = [&](int rows, double* dst) {
    return cudaMemset2DAsync(dst, sizeof(double) * ld_gf, 0, sizeof(double) * K, rows, ctx->stream);
  };
  fold(s->cellmass, 1, 0, Gf_out + (int64_t)Mtot * ld_gf);
  fold(s->cellmass2, 1, 0, lo + (int64_t)Mtot * ld_gf);
  if (s->obj) {
    fold(s->cellobj, 1, 0, Gf_out + (int64_t)(Mtot + 1) * ld_gf);
    fold(s->cellobj2, 1, 0, lo + (int64_t)(Mtot + 1) * ld_gf);
  } else {
    BASQ_CUDA(zero(1, Gf_out + (int64_t)(Mtot + 1) * ld_gf));
    BASQ_CUDA(zero(1, lo + (int64_t)(Mtot + 1) * ld_gf));
  }
  if (s->G2.p) fold(s->G2, Mtot, s->ldg, lo);
  else BASQ_CUDA(zero(Mtot, lo));
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

// out[r, i] = hi[r, i] + lo[r, i]: the one rounding from the exact hi and lo sums to the columns that are projected
__global__ void add_parts_kernel(const double* __restrict__ hi, const double* __restrict__ lo, int64_t ld, int rows,
                                 int K, double* __restrict__ out, int64_t ldo) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)rows * K) return;
  const int r = (int)(t / K), i = (int)(t % K);
  out[(int64_t)r * ldo + i] = __dadd_rn(hi[(int64_t)r * ld + i], lo[(int64_t)r * ld + i]);
}

// Reproducible sessions: the level system from the columns of session_level_fold_exact summed over every rank -
// the whole projection on every rank, with the same function and shapes as a single-GPU session.
int session_level_project_exact(basq_session* s, int lvl, int K, const int* node_host, const int* ppos_host,
                                const double* fpar_host, const double* Gf, int64_t ld_gf, double* A_out) {
  BASQ_CHECK(s->repro && s->Gc.p, BASQ_ERR_INVALID,
             "level_project_exact: the session is not reproducible (basq_ctx_reproducible) or has no pass");
  basq_ctx* ctx = s->ctx;
  const int rows = s->Mtot + 2;
  add_parts_kernel<<<(unsigned)ceil_div64((int64_t)rows * K, 256), 256, 0, ctx->stream>>>(
      Gf, Gf + (int64_t)rows * ld_gf, ld_gf, rows, K, s->Gc.as<double>(), K);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return session_level_project(s, lvl, K, node_host, ppos_host, fpar_host, s->Gc.as<double>(), K, 0, s->Mtot, A_out,
                               true);
}

int session_level(basq_session* s, int lvl, int K, const int* node_host, const int* ppos_host,
                  const double* fpar_host, double* A_out) {
  if (s->repro) {
    BASQ_TRY(session_level_fold_exact(s, lvl, K, node_host, s->Gf.as<double>(), s->S));
    return session_level_project_exact(s, lvl, K, node_host, ppos_host, fpar_host, s->Gf.as<double>(), s->S, A_out);
  }
  const int cnt = s->pass_F >> lvl;
  bool identity = (cnt == 1 && lvl == 0);  // plain round: the sets ARE the cells, project G as it is
  for (int i = 0; identity && i < K; ++i) identity = node_host[i] == i;
  if (identity)
    return session_level_project(s, lvl, K, node_host, ppos_host, fpar_host, s->G.as<double>(), s->ldg, 0, s->Mtot, A_out);
  BASQ_TRY(session_level_fold(s, lvl, K, node_host, s->Gf.as<double>(), s->S));
  return session_level_project(s, lvl, K, node_host, ppos_host, fpar_host, s->Gf.as<double>(), s->S, 0, s->Mtot, A_out);
}

// Host bookkeeping of a pass's level tree, shared by the single-call loop (recombine_impl) and
// mirrored by basq_b200/sharded.py: which nodes are presented to the next Caratheodory level.
struct LevelTree {
  int S = 0, F = 1, L = 0, lvl = 0;
  std::vector<int> act;      // node id of every column of the current level
  std::vector<double> fac;   // factor of every column's parent (1 at level 0)
  std::vector<int> node, ppos;
  std::vector<double> fpar;  // arguments of session_level for the current level
  void begin(int S_, int F_, int64_t R_glob) {
    S = S_; F = F_; lvl = 0; L = 0;
    while ((1 << L) < F) ++L;
    const int S0 = (int)std::min<int64_t>(S, R_glob);
    node.resize(S0); ppos.assign(S0, 0); fpar.assign(S0, 1.0);
    for (int j = 0; j < S0; ++j) node[j] = j;
    act = node; fac = fpar;
  }
  int columns() const { return (int)act.size(); }
  // consume the level's factors om[columns()] (1 = untouched); returns false after the last level,
  // when factor_host[F * S] has received the product of the factors along every surviving path
  bool advance(const double* om, double* factor_host, int* kept_out) {
    const int C = columns();
    const int stride = S << lvl;
    std::vector<int> nnode, nppos;
    std::vector<double> nfpar;
    for (int i = 0; i < C; ++i) {
      const double f = fac[i] * om[i];
      if (!(om[i] > 0.0) || !(f > 0.0)) continue;
      if (lvl < L) { nnode.push_back(act[i]); nppos.push_back(i); nfpar.push_back(f); }
      else factor_host[act[i]] = f;
      ++*kept_out;
    }
    if (lvl == L) return false;
    node.swap(nnode); ppos.swap(nppos); fpar.swap(nfpar);
    const int K = (int)node.size();
    act.resize(2 * K); fac.resize(2 * K);
    for (int i = 0; i < K; ++i) {
      act[i] = node[i]; act[K + i] = node[i] + stride;
      fac[i] = fac[K + i] = fpar[i];
    }
    ++lvl;
    return true;
  }
};

// columns of A (ld) selected by pick[t] and scaled by scale[t]: out[r, t] = scale[t] * A[r, pick[t]]
__global__ void gather_scaled_kernel(const double* __restrict__ A, int64_t ld, int rows, int K, const int* __restrict__ pick,
                                     const double* __restrict__ scale, double* __restrict__ out, int64_t ldo) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)rows * K) return;
  const int r = (int)(t / K), i = (int)(t % K);
  out[(int64_t)r * ldo + i] = scale[i] * A[(int64_t)r * ld + pick[i]];
}

// One Caratheodory level with the objective row of SOBER/_rchq.py:67-69,138-146,177-196.
// A [n + 1, C] (ld): rows 0..n-1 the moment system, row n the objective sums (obj = -calc_obj, so the
// rule's expected calc_obj goes UP when sum_t omega_t A[n, t] goes down).  Step 1: Caratheodory on all
// n + 1 rows keeps <= n + 1 columns and their objective value.  Step 2 (:177-196): the kept columns
// have a one-dimensional null space with respect to the n moment rows; move along it in the
// direction that does not increase the objective row until one more column drops: <= n columns
// survive, the n moments are preserved exactly, the objective is at least as good as the measure's.
// omega_out [C] (device) receives the final relative factors.  A is destroyed.
int car_with_objective(basq_ctx* ctx, double* A, int n, int C, int lda, double* omega_out) {
  DevBuf copy, dpick, dscale;
  BASQ_TRY(copy.alloc(ctx, sizeof(double) * (size_t)(n + 1) * lda));
  BASQ_CUDA(cudaMemcpyAsync(copy.p, A, sizeof(double) * (size_t)(n + 1) * lda, cudaMemcpyDeviceToDevice, ctx->stream));
  BASQ_TRY(caratheodory(ctx, A, n + 1, C, lda, omega_out));
  std::vector<double> om(C), objrow(C);
  BASQ_CUDA(cudaMemcpyAsync(om.data(), omega_out, sizeof(double) * C, cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaMemcpyAsync(objrow.data(), copy.as<double>() + (int64_t)n * lda, sizeof(double) * C,
                            cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  BASQ_TRY(check_finite_host(om.data(), C, "omega"));
  std::vector<int> pick;
  std::vector<double> scale;
  for (int i = 0; i < C; ++i)
    if (om[i] > 0.0) { pick.push_back(i); scale.push_back(om[i]); }
  const int K = (int)pick.size();
  if (K <= n) return BASQ_OK;  // already small enough (rank-deficient system)
  BASQ_CHECK(K == n + 1, BASQ_ERR_NUMERIC, "objective step: %d columns survive a system of %d rows", K, n + 1);
  BASQ_TRY(dpick.alloc(ctx, sizeof(int) * K));
  BASQ_TRY(dscale.alloc(ctx, sizeof(double) * K));
  BASQ_CUDA(cudaMemcpyAsync(dpick.p, pick.data(), sizeof(int) * K, cudaMemcpyHostToDevice, ctx->stream));
  BASQ_CUDA(cudaMemcpyAsync(dscale.p, scale.data(), sizeof(double) * K, cudaMemcpyHostToDevice, ctx->stream));
  gather_scaled_kernel<<<(unsigned)ceil_div64((int64_t)n * K, 256), 256, 0, ctx->stream>>>(
      copy.as<double>(), lda, n, K, dpick.as<int>(), dscale.as<double>(), A, lda);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  DevBuf om2;
  BASQ_TRY(om2.alloc(ctx, sizeof(double) * K));
  BASQ_TRY(caratheodory(ctx, A, n, K, lda, om2.as<double>()));
  std::vector<double> w2(K);
  BASQ_CUDA(cudaMemcpyAsync(w2.data(), om2.p, sizeof(double) * K, cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  BASQ_TRY(check_finite_host(w2.data(), K, "omega (objective step)"));
  // null direction v = 1 - w2 of the scaled columns; d = its objective slope
  double d = 0.0;
  for (int t = 0; t < K; ++t) d += (1.0 - w2[t]) * scale[t] * objrow[pick[t]];
  std::vector<double> rho(K);
  if (d >= 0.0) {
    rho = w2;  // moving by -v lowers (or keeps) the objective row: the step the kernel took
  } else {
    double beta = -1.0;
    int arg = -1;
    for (int t = 0; t < K; ++t) {
      const double v = 1.0 - w2[t];
      if (v < 0.0 && (arg < 0 || 1.0 / (-v) < beta)) { beta = 1.0 / (-v); arg = t; }
    }
    if (arg < 0) {
      rho = w2;  // the direction has no negative entry: only the kernel's side reaches a face
    } else {
      for (int t = 0; t < K; ++t) rho[t] = std::max(0.0, 1.0 + beta * (1.0 - w2[t]));
      rho[arg] = 0.0;
    }
  }
  for (int i = 0; i < C; ++i) om[i] = 0.0;
  for (int t = 0; t < K; ++t) om[pick[t]] = scale[t] * rho[t];
  BASQ_CUDA(cudaMemcpyAsync(omega_out, om.data(), sizeof(double) * C, cudaMemcpyHostToDevice, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

// All levels of the current pass for a single rank: factor_host[F * S] out.
int session_pass_levels(basq_session* s, double* A, double* omega_dev, double* factor_host) {
  basq_ctx* ctx = s->ctx;
  const int n = s->n, S = s->S, F = s->pass_F;
  for (int c = 0; c < F * S; ++c) factor_host[c] = 0.0;
  LevelTree tree;
  tree.begin(S, F, s->pass_R);
  std::vector<double> om(S);
  for (;;) {
    const int K = (int)tree.node.size();
    BASQ_CHECK(K >= 1, BASQ_ERR_NUMERIC, "pass: no active node at level %d", tree.lvl);
    const int C = tree.columns();
    if (C > n) {
      BASQ_TRY(session_level(s, tree.lvl, K, tree.node.data(), tree.ppos.data(), tree.fpar.data(), A));
      if (s->obj) BASQ_TRY(car_with_objective(ctx, A, n, C, S, omega_dev));
      else BASQ_TRY(caratheodory(ctx, A, n, C, S, omega_dev));
      BASQ_CUDA(cudaMemcpyAsync(om.data(), omega_dev, sizeof(double) * C, cudaMemcpyDeviceToHost, ctx->stream));
      BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
      BASQ_TRY(check_finite_host(om.data(), C, "omega"));
    } else {
      // nothing to eliminate at this level; deeper levels still need this level's raw columns
      if (tree.lvl < tree.L)
        BASQ_TRY(session_level(s, tree.lvl, K, tree.node.data(), tree.ppos.data(), tree.fpar.data(), A));
      for (int i = 0; i < C; ++i) om[i] = 1.0;
    }
    int kept = 0;
    const int lvl = tree.lvl;
    const bool more = tree.advance(om.data(), factor_host, &kept);
    BASQ_CHECK(kept >= 1, BASQ_ERR_NUMERIC, "pass: the Caratheodory step kept no set (level %d)", lvl);
    if (!more) break;
  }
  return BASQ_OK;
}

// Rescale the kept cells by factor_host[F * S] (0 = dropped), drop the rest, compact in order.
int session_apply_impl(basq_session* s, int64_t R_glob, int64_t off, int F, const double* factor_host,
                       int64_t* R_loc_new) {
  basq_ctx* ctx = s->ctx;
  PhaseTimer t(ctx, PH_APPLY);
  const int cells = F * s->S;
  const int c_eff = (int)std::min<int64_t>(cells, R_glob);
  BASQ_TRY(session_reserve_cells(s, cells));
  BASQ_TRY(check_finite_host(factor_host, c_eff, "omega"));
  int K = 0;
  for (int j = 0; j < cells; ++j) {
    s->rank_host[j] = K;
    s->omega_host[j] = (j < c_eff && factor_host[j] > 0.0) ? factor_host[j] : 0.0;
    if (s->omega_host[j] > 0.0) ++K;
  }
  BASQ_CHECK(K >= 1, BASQ_ERR_NUMERIC, "apply: the Caratheodory step kept no set");
  auto D = [&](int64_t g) {  // kept points among global positions < g
    const int64_t e = g / cells;
    const int j = (int)(g % cells);
    return e * (int64_t)K + s->rank_host[j];
  };
  const int64_t dest_base = D(off);
  const int64_t new_count = D(off + s->pool.count) - dest_base;
  DevBuf dom;
  BASQ_TRY(dom.alloc(ctx, sizeof(double) * (size_t)cells));
  BASQ_CUDA(cudaMemcpyAsync(dom.p, s->omega_host.data(), sizeof(double) * cells, cudaMemcpyHostToDevice, ctx->stream));
  BASQ_CUDA(cudaMemcpyAsync(s->rank.p, s->rank_host.data(), sizeof(int) * cells, cudaMemcpyHostToDevice, ctx->stream));
  BASQ_TRY(apply_round(ctx, &s->pool, off, cells, dom.as<double>(), s->rank.as<int>(), K, s->scale_wf, dest_base,
                       new_count));
  // the host tables are reused by the next pass: make sure the H2D copies have consumed them
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  if (R_loc_new) *R_loc_new = new_count;
  return BASQ_OK;
}

// Cell factor of a pass over R_glob points (at most R_loc_max on one rank).  A pass with F = 2^L
// costs one sweep of Mtot * R_loc kernel evaluations (tiles of 32 members per cell: short cells
// waste slots) plus (1 + L/2) projections of S columns, and replaces L + 1 rounds: pick the F with
// the lowest cost per level.  One evaluation ~ 4.4 fp64-GEMM flop at the measured kernel rates.
int choose_cell_factor(const basq_session* s, int64_t R_glob, int64_t R_loc_max) {
  if (s->repro) R_loc_max = R_glob;   // the cells must not depend on how the points are split over ranks
  static const int forced = [] { const char* e = getenv("BASQ_CELL_FACTOR"); return e ? atoi(e) : 0; }();
  const int64_t S = s->S;
  auto fits = [&](int f) { return R_glob >= (int64_t)4 * f * S; };
  if (s->nl != NL_LIN && forced < 1) {
    // pairwise non-linear kernels (WSABI-M, MMLT): a sweep costs an extra 2 n_obs M fp64 flop per
    // candidate (the posterior correction per pair), far more than any projection: refine as far as
    // the cells keep a handful of members
    int F = 1;
    while (F * 2 <= BASQ_MAX_CELL_FACTOR && fits(F * 2) && R_loc_max >= (int64_t)8 * F * 2 * S) F *= 2;
    return F;
  }
  if (forced >= 1) {
    int F = 1;
    while (F * 2 <= forced && F * 2 <= BASQ_MAX_CELL_FACTOR && fits(F * 2)) F *= 2;
    return F;
  }
  const double proj = 2.0 * s->q * (double)S / 4.4;  // one projection of S columns, in evaluations per landmark
  int best = 1;
  double best_cost = 0.0;
  for (int F = 1, L = 0; F <= BASQ_MAX_CELL_FACTOR; F *= 2, ++L) {
    if (F > 1 && !fits(F)) break;
    const double members = (double)R_loc_max / ((double)F * S);          // local members per cell
    const double slots = 32.0 * ceil(std::max(members, 1e-9) / 32.0);    // tile slots they occupy
    const double cost = ((double)R_loc_max * (slots / std::max(members, 1e-9)) + proj * (1.0 + 0.5 * L)) / (L + 1);
    if (F == 1 || cost < best_cost) { best = F; best_cost = cost; }
  }
  return best;
}

// Grids of a reproducible pass over R_glob live points from the maxima over every rank of |wf|, |mu| and |mu obj|
// (record_maxima, max-reduced over the ranks: exact).  A bound B on the sum of |terms| of every set sum, mass and
// objective sum gives Q = 2^(ceil(log2 B) - 51): every term is below 2^51 Q and every partial sum below 2^53 Q.
//   linear modes: |wf_p k| <= |wf_p| sigma_f^2          (wf = mu, or mu m(x) for WSABI-L)
//   WSABI-M:      |mu_p (sz C sx_p + C^2 / 2)| <= |mu_p| (max|sz| sigma_f^2 |sx_p| + sigma_f^4 / 2)   (|C| <= sigma_f^2)
//   MMLT:         |mu_p sz sx_p expm1(C)| <= |mu_p| max|sz| |sx_p| max(expm1(sigma_f^2), 1)
int session_set_grid(basq_session* s, int64_t R_glob, const double* mx) {
  BASQ_CHECK(s->repro, BASQ_ERR_INVALID, "set_grid: the session is not reproducible (basq_ctx_reproducible)");
  BASQ_CHECK(R_glob >= 1, BASQ_ERR_INVALID, "set_grid: R_glob must be positive");
  const double os = s->kp.outputscale, R = (double)R_glob;
  double B[3];
  if (s->nl == NL_WSABIM) B[0] = R * mx[1] * (s->szmax * os * mx[0] + 0.5 * os * os);
  else if (s->nl == NL_MMLT) B[0] = R * mx[1] * s->szmax * mx[0] * std::max(expm1(os), 1.0);
  else B[0] = R * mx[0] * os;
  B[1] = R * mx[1];
  B[2] = R * mx[2];
  // Second grids for the remainders term - hi (each below Q / 2, so their sum is below R Q / 2): the fp64 terms,
  // masses and objective sums keep their fp64 accuracy, about 2^-103 R^2 B absolute.
  for (int i = 0; i < 3; ++i) {
    BASQ_CHECK(isfinite(B[i]) && B[i] < 0x1p1000, BASQ_ERR_NUMERIC, "set_grid: weights or factors out of range");
    grid_pair(B[i], R, &s->grid_m[i], &s->grid_m2[i]);
  }
  s->grid_R = R_glob;
  return BASQ_OK;
}

int session_grid_local(basq_session* s, double* max_host) {
  BASQ_CHECK(s->repro, BASQ_ERR_INVALID, "grid_maxima: the session is not reproducible (basq_ctx_reproducible)");
  return record_maxima(s->ctx, s->pool, s->obj, max_host);
}

// Phi[p_lo..p_hi, q] for the session's live records
int session_features(basq_session* s, double* Phi_out) {
  basq_ctx* ctx = s->ctx;
  const int64_t N = s->pool.count;
  const int64_t P = 16384;
  DevBuf Gc;
  BASQ_TRY(Gc.alloc(ctx, sizeof(double) * (size_t)s->Mtot * P));
  for (int64_t p0 = 0; p0 < N; p0 += P) {
    const int64_t p1 = std::min(N, p0 + P);
    BASQ_TRY(session_set_sums(s, -p0, (int)P, p0, p1, Gc.as<double>(), P));
    // Phi[p0 + j, i] = sum_m G[m, j] U'[i, m]
    BASQ_TRY(dgemm(ctx, true, true, (int)(p1 - p0), s->q, s->Mtot, 1.0, Gc.as<double>(), P, s->Uprime.as<double>(),
                   s->Mtot, 0.0, Phi_out + p0 * s->q, s->q));
  }
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

int recombine_impl(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N, const void* Z, int64_t M,
                   const double* U, int q, const double* mu, int64_t* idx_out, double* w_out, int* n_out_host,
                   const double* obj = nullptr) {
  BASQ_CHECK(idx_out && w_out && n_out_host, BASQ_ERR_INVALID, "recombine: NULL output");
  std::unique_ptr<basq_session> s(new (std::nothrow) basq_session());
  BASQ_CHECK(s, BASQ_ERR_INVALID, "out of host memory");
  trace_point(ctx, "recombine: enter");
  BASQ_TRY(session_create_impl(ctx, desc, X, N, N, 0, Z, M, U, q, mu, 0, s.get()));
  trace_point(ctx, "recombine: session created");
  const int n = s->n, S = s->S;
  if (obj) { s->obj = obj; s->rows = n + 1; }
  DevBuf A, omega;
  BASQ_TRY(A.alloc(ctx, sizeof(double) * (size_t)(n + 1) * S));
  BASQ_TRY(omega.alloc(ctx, sizeof(double) * S));
  int64_t R = s->pool.count;
  std::vector<double> factor;
  int rounds = 0;
  while (R > n) {
    BASQ_CHECK(++rounds <= 256, BASQ_ERR_NUMERIC, "recombine: no convergence after 256 passes");
    const int F = choose_cell_factor(s.get(), R, R);
    factor.resize((size_t)F * S);
    if (s->repro) {
      double mx[3];
      BASQ_TRY(session_grid_local(s.get(), mx));
      BASQ_TRY(session_set_grid(s.get(), R, mx));
    }
    BASQ_TRY(session_pass_begin(s.get(), R, 0, F));
    trace_point(ctx, "  pass: set sums");
    BASQ_TRY(session_pass_levels(s.get(), A.as<double>(), omega.as<double>(), factor.data()));
    trace_point(ctx, "  pass: caratheodory levels");
    int64_t Rn = 0;
    BASQ_TRY(session_apply_impl(s.get(), R, 0, F, factor.data(), &Rn));
    trace_point(ctx, "  pass: apply");
    BASQ_CHECK(Rn < R, BASQ_ERR_NUMERIC, "recombine: pass %d made no progress (%lld points)", rounds, (long long)R);
    R = Rn;
  }
  trace_point(ctx, "recombine: rounds done");
  BASQ_TRY(extract_result(ctx, s->pool, 0, idx_out, w_out));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  *n_out_host = (int)R;
  return BASQ_OK;
}

}  // namespace
}  // namespace basq

// =============================================================================================
// extern "C"
// =============================================================================================
extern "C" {

int basq_abi_version(void) { return BASQ_ABI_VERSION; }
const char* basq_last_error(void) { return basq::last_error_cstr(); }

int basq_ctx_create(int device, void* stream, basq_ctx** out) {
  BASQ_CHECK(out != nullptr, BASQ_ERR_INVALID, "basq_ctx_create: out is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error("no CUDA device available (%s); basq_b200 has no CPU fallback",
              e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    return BASQ_ERR_CUDA;
  }
  BASQ_CHECK(device >= 0 && device < ndev, BASQ_ERR_INVALID, "device %d out of range (have %d)", device, ndev);
  BASQ_CUDA(cudaSetDevice(device));
  basq_ctx* c = new (std::nothrow) basq_ctx();
  BASQ_CHECK(c, BASQ_ERR_INVALID, "out of host memory");
  c->device = device;
  c->stream = reinterpret_cast<cudaStream_t>(stream);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
    delete c;
    set_error("cudaGetDeviceProperties failed");
    return BASQ_ERR_CUDA;
  }
  c->num_sms = prop.multiProcessorCount;
  c->smem_optin = prop.sharedMemPerBlockOptin;
  if (prop.major < 10) {
    delete c;
    set_error("basq_b200 is built for sm_100a (Blackwell B200); device %d is sm_%d%d", device, prop.major, prop.minor);
    return BASQ_ERR_CUDA;
  }
  // Scratch memory comes from the context's own block cache (common.cuh).  Automatic trimming at the end of every
  // top-level call is opt-in (BASQ_POOL_KEEP_MB): a trim is followed by re-allocation at driver speed.
  c->pool_keep = UINT64_MAX;
  if (const char* t = getenv("BASQ_POOL_KEEP_MB")) c->pool_keep = (uint64_t)strtoull(t, nullptr, 10) << 20;
  { const char* t = getenv("BASQ_TRACE"); c->trace = t && t[0] == '1'; }
  { const char* t = getenv("BASQ_CAR_GENERAL"); c->force_general_car = t && t[0] == '1'; }
  { const char* t = getenv("BASQ_F32_KAPPA_MAX"); if (t) c->kappa_max = atof(t); }
  { const char* t = getenv("BASQ_F64_EVAL_F32"); c->eval_f32 = t && t[0] == '1'; }
  *out = c;
  return BASQ_OK;
}

void basq_ctx_destroy(basq_ctx* ctx) {
  if (!ctx) return;
  ctx->resolve_spans();
  for (cudaEvent_t e : ctx->free_events) cudaEventDestroy(e);
  if (ctx->stage || ctx->side) cudaStreamSynchronize(ctx->stream);
  if (ctx->side) {
    cudaStreamSynchronize(ctx->side);
    cudaStreamDestroy(ctx->side);
  }
  for (cudaEvent_t e : ctx->side_ev)
    if (e) cudaEventDestroy(e);
  if (ctx->stage) cudaFreeHost(ctx->stage);
  if (ctx->host_x) cudaFree(ctx->host_x);
  for (cudaEvent_t e : ctx->stage_ev)
    if (e) cudaEventDestroy(e);
  ctx->block_trim(0);
  (void)cudaGetLastError();
  delete ctx;
}

int basq_ctx_trim(basq_ctx* ctx, int64_t keep_bytes) {
  BASQ_CHECK(ctx, BASQ_ERR_INVALID, "ctx is NULL");
  if (keep_bytes >= 0 && ctx->host_x) {   // an explicit request also drops the candidate buffer of basq_recombine_host
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
    BASQ_CUDA(cudaFree(ctx->host_x));
    ctx->host_x = nullptr;
    ctx->host_x_bytes = 0;
  }
  const uint64_t keep = keep_bytes < 0 ? ctx->pool_keep : (uint64_t)keep_bytes;
  if (keep == UINT64_MAX) return BASQ_OK;
  ctx->block_trim((size_t)keep);
  return BASQ_OK;
}

int basq_ctx_memory(const basq_ctx* ctx, uint64_t* cached_bytes_host, uint64_t* live_bytes_host,
                    int64_t* driver_allocs_host) {
  BASQ_CHECK(ctx, BASQ_ERR_INVALID, "ctx is NULL");
  if (cached_bytes_host) *cached_bytes_host = ctx->cached_bytes + ctx->host_x_bytes;
  if (live_bytes_host) *live_bytes_host = ctx->live_bytes;
  if (driver_allocs_host) *driver_allocs_host = ctx->driver_allocs;
  return BASQ_OK;
}

int64_t basq_ctx_launch_count(const basq_ctx* ctx) { return ctx ? ctx->launches : 0; }

int basq_ctx_allow_f32_eval(basq_ctx* ctx, int on, int64_t* demotions_host) {
  BASQ_CHECK(ctx, BASQ_ERR_INVALID, "basq_ctx_allow_f32_eval: NULL context");
  if (on >= 0) ctx->eval_f32 = on != 0;
  if (demotions_host) *demotions_host = ctx->demotions;
  return BASQ_OK;
}

int basq_ctx_reproducible(basq_ctx* ctx, int on) {
  BASQ_CHECK(ctx, BASQ_ERR_INVALID, "basq_ctx_reproducible: NULL context");
  if (on >= 0) ctx->reproducible = on != 0;
  return BASQ_OK;
}

int basq_ctx_set_seed(basq_ctx* ctx, uint64_t seed) {
  BASQ_CHECK(ctx, BASQ_ERR_INVALID, "basq_ctx_set_seed: NULL context");
  ctx->seed = seed;
  ctx->draws = 0;
  return BASQ_OK;
}

int basq_ctx_conditioning(basq_ctx* ctx, double kappa_max, double* last_kappa_host, int64_t* promotions_host) {
  BASQ_CHECK(ctx, BASQ_ERR_INVALID, "ctx is NULL");
  if (kappa_max >= 0.0) ctx->kappa_max = kappa_max;
  if (last_kappa_host) *last_kappa_host = ctx->last_kappa;
  if (promotions_host) *promotions_host = ctx->promotions;
  return BASQ_OK;
}
int64_t basq_ctx_pair_evals(const basq_ctx* ctx) { return ctx ? ctx->pair_evals : 0; }

int basq_ctx_profile(basq_ctx* ctx, int enable) {
  BASQ_CHECK(ctx, BASQ_ERR_INVALID, "ctx is NULL");
  if (!enable) ctx->resolve_spans();
  ctx->profile = enable != 0;
  return BASQ_OK;
}

int basq_ctx_profile_read(basq_ctx* ctx, double* ms_host, int64_t* calls_host, int reset) {
  BASQ_CHECK(ctx && ms_host, BASQ_ERR_INVALID, "NULL argument");
  ctx->resolve_spans();
  for (int i = 0; i < PH_COUNT; ++i) {
    ms_host[i] = ctx->phase_ms[i];
    if (calls_host) calls_host[i] = ctx->phase_calls[i];
    if (reset) {
      ctx->phase_ms[i] = 0.0;
      ctx->phase_calls[i] = 0;
    }
  }
  return BASQ_OK;
}

int basq_dgemm(basq_ctx* ctx, int transA, int transB, int m, int n, int k, double alpha, const double* A, int lda,
               const double* B, int ldb, double beta, double* C, int ldc) {
  BASQ_CHECK(ctx && A && B && C, BASQ_ERR_INVALID, "basq_dgemm: NULL argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  return dgemm(ctx, transA != 0, transB != 0, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc);
}

int basq_tgemm(basq_ctx* ctx, int m, int n, int k, const double* A, int lda, const double* B, int ldb, double* C,
               int ldc) {
  BASQ_CHECK(ctx && A && B && C, BASQ_ERR_INVALID, "basq_tgemm: NULL argument");
  BASQ_CHECK(m >= 1 && n >= 1 && k >= 1 && lda >= k && ldb >= k && ldc >= n, BASQ_ERR_INVALID, "basq_tgemm: bad shape");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  BlkOperand a, b;
  BASQ_TRY(a.alloc(ctx, m, k));
  BASQ_TRY(b.alloc(ctx, n, k));
  BASQ_TRY(blk_from_f64(ctx, A, lda, false, &a));
  BASQ_TRY(blk_from_f64(ctx, B, ldb, false, &b));
  BASQ_TRY(tgemm(ctx, a, b, 1.0, C, ldc, false));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

int basq_igemm(basq_ctx* ctx, int m, int n, int k, const double* A, int lda, int row0, int nrows, const double* B,
               int ldb, double* C, int ldc, int accumulate) {
  BASQ_CHECK(ctx && A && B && C, BASQ_ERR_INVALID, "basq_igemm: NULL argument");
  BASQ_CHECK(m >= 1 && n >= 1 && k >= 1 && lda >= k && row0 >= 0 && nrows >= 1 && row0 + nrows <= k && ldb >= n &&
                 ldc >= n,
             BASQ_ERR_INVALID, "basq_igemm: bad shape");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  DigOperand a, b;
  BASQ_TRY(dig_from_f64(ctx, A, lda, false, m, k, 0, 128, &a));
  BASQ_TRY(dig_from_f64(ctx, B, ldb, true, n, nrows, row0, 64, &b));
  BASQ_TRY(igemm(ctx, a, b, 1.0, C, ldc, accumulate != 0));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

int basq_gram(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t a, const void* Y, int64_t b,
              double* out) {
  BASQ_CHECK(ctx && desc && X && Y && out, BASQ_ERR_INVALID, "basq_gram: NULL argument");
  BASQ_CHECK(a >= 1 && b >= 1, BASQ_ERR_INVALID, "basq_gram: empty operand");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  const int rc = basq::gram_matrix(ctx, desc, X, a, Y, b, out, false);
  basq_ctx_trim(ctx, -1);
  return rc;
}

}  // extern "C"

// kernel(X, Y) [a, b] in fp64.  tensor_correction: the posterior-covariance correction
// (K_xX W) K_Xy - an [a, n_obs] x [n_obs, b] product - runs on the tensor cores with fp32 accuracy
// (tgemm.cu).  Only the Nystrom range finder asks for that: its products with this matrix are
// fp32-accurate split products as well, and only the span of the resulting basis matters.
int basq::gram_matrix(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t a, const void* Y, int64_t b,
                      double* out, bool tensor_correction, int64_t diag_col0) {
  KParams kp;
  BASQ_TRY(make_kparams(desc, &kp));
  BASQ_TRY(compute_center(ctx, desc, X, a, &kp));
  Landmarks lmx;
  BASQ_TRY(prep_landmarks(ctx, kp, desc->dtype, X, a, nullptr, 0, &lmx));
  BASQ_TRY(base_gram(ctx, kp, lmx.view(), Y, b, out, b));
  const int mode = desc->mode;
  if (mode != BASQ_PLAIN) {
    const int n_obs = desc->n_obs;
    Landmarks lmobs;
    BASQ_TRY(prep_landmarks(ctx, kp, desc->dtype, desc->Xobs, n_obs, nullptr, 0, &lmobs));
    DevBuf KxX, T, KXy, fx, fy;
    BASQ_TRY(KxX.alloc(ctx, sizeof(double) * (size_t)a * n_obs));
    BASQ_TRY(T.alloc(ctx, sizeof(double) * (size_t)a * n_obs));
    BASQ_TRY(KXy.alloc(ctx, sizeof(double) * (size_t)n_obs * b));
    BASQ_TRY(base_gram(ctx, kp, lmx.view(), desc->Xobs, n_obs, KxX.as<double>(), n_obs));
    BASQ_TRY(base_gram(ctx, kp, lmobs.view(), Y, b, KXy.as<double>(), b));
    BASQ_CHECK(a < (1ll << 31) && b < (1ll << 31), BASQ_ERR_UNSUPPORTED, "basq_gram: operand too large");
    BASQ_TRY(dgemm(ctx, false, false, (int)a, n_obs, n_obs, 1.0, KxX.as<double>(), n_obs, desc->W, n_obs, 0.0,
                   T.as<double>(), n_obs));
    if (tensor_correction && desc->dtype == BASQ_F32) {
      BlkOperand Tb, Yb;
      BASQ_TRY(Tb.alloc(ctx, (int)a, n_obs));
      BASQ_TRY(Yb.alloc(ctx, (int)b, n_obs));
      BASQ_TRY(blk_from_f64(ctx, T.as<double>(), n_obs, false, &Tb));
      BASQ_TRY(blk_from_f64(ctx, KXy.as<double>(), b, true, &Yb));   // K_Xy^T as [b, n_obs] operand
      BASQ_TRY(tgemm(ctx, Tb, Yb, -1.0, out, b, false, /*accumulate=*/true));
      BASQ_CUDA(cudaStreamSynchronize(ctx->stream));                 // operands go out of scope
    } else {
      BASQ_TRY(dgemm(ctx, false, false, (int)a, (int)b, n_obs, -1.0, T.as<double>(), n_obs, KXy.as<double>(), b, 1.0,
                     out, b));
    }
    const bool warped = (mode == BASQ_WSABI_L || mode == BASQ_WSABI_M || mode == BASQ_MMLT_G);
    if (warped) {
      BASQ_TRY(fx.alloc(ctx, sizeof(double) * a));
      BASQ_TRY(fy.alloc(ctx, sizeof(double) * b));
      BASQ_TRY(warp_factor(ctx, desc, kp, lmobs.view(), X, a, fx.as<double>()));
      BASQ_TRY(warp_factor(ctx, desc, kp, lmobs.view(), Y, b, fy.as<double>()));
    }
    const double pre_add = desc->noise_diag ? desc->noise : 0.0;
    if (warped || desc->diag_add != 0.0 || pre_add != 0.0) {
      const int64_t tot = a * b;
      warp_gram_kernel<<<(unsigned)ceil_div64(tot, 256), 256, 0, ctx->stream>>>(
          out, a, b, warped ? mode : BASQ_PRED_COV, fx.as<double>(), fy.as<double>(), pre_add, desc->diag_add, diag_col0);
      ctx->launches++;
      BASQ_CUDA(cudaGetLastError());
    }
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  } else if (desc->diag_add != 0.0) {
    const int64_t tot = a * b;
    warp_gram_kernel<<<(unsigned)ceil_div64(tot, 256), 256, 0, ctx->stream>>>(out, a, b, BASQ_PLAIN, nullptr, nullptr,
                                                                             0.0, desc->diag_add, diag_col0);
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
  }
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

extern "C" {

int basq_gp_predict(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N, int space, double offset,
                    double* mean_out, double* var_out) {
  BASQ_CHECK(ctx && desc && X && mean_out, BASQ_ERR_INVALID, "basq_gp_predict: NULL argument");
  BASQ_CHECK(desc->n_obs > 0 && desc->Xobs && desc->W && desc->alpha, BASQ_ERR_INVALID,
             "basq_gp_predict needs the GP caches (n_obs, Xobs, W, alpha)");
  const bool need_var = var_out != nullptr || (space == 1 && (desc->mode == BASQ_WSABI_M || desc->mode == BASQ_MMLT_G));
  // the limit of the fp32 variance route, checked again in gp_variance_tc: here before anything is allocated
  BASQ_CHECK(!(need_var && N > 0 && gpvar_route(ctx, desc)) || desc->n_obs <= GPV_MAX_OBS, BASQ_ERR_UNSUPPORTED,
             "basq_gp_predict: %d observations; the fp32 posterior variance takes at most %d", desc->n_obs, GPV_MAX_OBS);
  BASQ_CUDA(cudaSetDevice(ctx->device));
  KParams kp;
  basq_kernel_desc d2 = *desc;
  if (d2.mode == BASQ_PLAIN) d2.mode = BASQ_PRED_COV;
  BASQ_TRY(make_kparams(&d2, &kp));
  BASQ_TRY(compute_center(ctx, &d2, d2.Xobs, d2.n_obs, &kp));
  Landmarks lmobs;
  BASQ_TRY(prep_landmarks(ctx, kp, d2.dtype, d2.Xobs, d2.n_obs, nullptr, 0, &lmobs));
  const bool warped = (desc->mode == BASQ_WSABI_L || desc->mode == BASQ_WSABI_M || desc->mode == BASQ_MMLT_G);
  DevBuf vtmp;
  double* var = var_out;
  if (need_var && !var) {
    BASQ_TRY(vtmp.alloc(ctx, sizeof(double) * N));
    var = vtmp.as<double>();
  }
  BASQ_TRY(gp_predict_impl(ctx, &d2, kp, lmobs.view(), X, N, mean_out, need_var ? var : nullptr));
  if (space == 1 && warped && N > 0) {
    model_space_kernel<<<(unsigned)ceil_div64(N, 256), 256, 0, ctx->stream>>>(desc->mode, offset, N, mean_out,
                                                                              need_var ? var : nullptr,
                                                                              var_out != nullptr ? 1 : 0);
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
  }
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

int basq_nystrom_basis(basq_ctx* ctx, const basq_kernel_desc* desc, const void* Z, int64_t M, int q,
                       const double* Omega, int niter, double* U_out, double* S_out) {
  BASQ_CHECK(ctx && desc && Z && U_out, BASQ_ERR_INVALID, "basq_nystrom_basis: NULL argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  const int rc = nystrom_basis(ctx, desc, Z, M, q, Omega, niter, U_out, S_out, nullptr);
  basq_ctx_trim(ctx, -1);
  return rc;
}

int basq_nystrom_basis_sharded(basq_ctx* ctx, const basq_kernel_desc* desc, const void* Z, int64_t M, int q,
                               const double* Omega, int niter, int rank, int world, double* gram_buf,
                               double* rows_buf, basq_exchange_fn exchange, void* user, double* U_out) {
  BASQ_CHECK(ctx && desc && Z && U_out && gram_buf && rows_buf && exchange, BASQ_ERR_INVALID,
             "basq_nystrom_basis_sharded: NULL argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  const NysShard shard{rank, world, exchange, user, gram_buf, rows_buf};
  const int rc = nystrom_basis(ctx, desc, Z, M, q, Omega, niter, U_out, nullptr, &shard);
  basq_ctx_trim(ctx, -1);
  return rc;
}

int basq_features(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N, const void* Z, int64_t M,
                  const double* U, int q, double* Phi_out) {
  BASQ_CHECK(ctx && desc && X && Z && U && Phi_out, BASQ_ERR_INVALID, "basq_features: NULL argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  std::unique_ptr<basq_session> s(new (std::nothrow) basq_session());
  BASQ_CHECK(s, BASQ_ERR_INVALID, "out of host memory");
  // unit weights: the feature of a point is its set sum with weight 1 (S = 4 keeps the round buffers tiny)
  DevBuf ones;
  BASQ_TRY(ones.alloc(ctx, sizeof(double) * N));
  {
    std::vector<double> h((size_t)N, 1.0);
    BASQ_CUDA(cudaMemcpyAsync(ones.p, h.data(), sizeof(double) * N, cudaMemcpyHostToDevice, ctx->stream));
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  BASQ_TRY(session_create_impl(ctx, desc, X, N, N, 0, Z, M, U, q, ones.as<double>(), 4, s.get()));
  const int rc = session_features(s.get(), Phi_out);
  s.reset();
  ones.release();
  basq_ctx_trim(ctx, -1);
  return rc;
}

int basq_car(basq_ctx* ctx, double* A, int n, int S, int lda, double* omega_out, int* n_kept_host) {
  BASQ_CHECK(ctx && A && omega_out, BASQ_ERR_INVALID, "basq_car: NULL argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  BASQ_TRY(caratheodory(ctx, A, n, S, lda, omega_out));
  if (n_kept_host) {
    std::vector<double> h((size_t)S);
    BASQ_CUDA(cudaMemcpyAsync(h.data(), omega_out, sizeof(double) * S, cudaMemcpyDeviceToHost, ctx->stream));
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
    int k = 0;
    for (double v : h) k += v > 0.0;
    *n_kept_host = k;
  }
  return BASQ_OK;
}

int basq_recombine(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N, const void* Z, int64_t M,
                   const double* U, int q, const double* mu, int64_t* idx_out, double* w_out, int* n_out_host) {
  BASQ_CHECK(ctx, BASQ_ERR_INVALID, "ctx is NULL");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  const int rc = recombine_impl(ctx, desc, X, N, Z, M, U, q, mu, idx_out, w_out, n_out_host);
  basq_ctx_trim(ctx, -1);
  return rc;
}

int basq_recombine_objective(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N, const void* Z,
                             int64_t M, const double* U, int q, const double* mu, const double* obj, int64_t* idx_out,
                             double* w_out, int* n_out_host) {
  BASQ_CHECK(ctx && obj, BASQ_ERR_INVALID, "basq_recombine_objective: NULL argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  const int rc = recombine_impl(ctx, desc, X, N, Z, M, U, q, mu, idx_out, w_out, n_out_host, obj);
  basq_ctx_trim(ctx, -1);
  return rc;
}

int basq_car_objective(basq_ctx* ctx, double* A, int n, int C, int lda, double* omega_out) {
  BASQ_CHECK(ctx && A && omega_out, BASQ_ERR_INVALID, "basq_car_objective: NULL argument");
  BASQ_CHECK(n >= 1 && C >= 1 && lda >= C, BASQ_ERR_INVALID, "basq_car_objective: bad shape");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  if (C <= n) return caratheodory(ctx, A, n, C, lda, omega_out);
  return car_with_objective(ctx, A, n, C, lda, omega_out);
}

int basq_session_set_objective(basq_session* s, const double* obj) {
  BASQ_CHECK(s, BASQ_ERR_INVALID, "NULL argument");
  s->obj = obj;
  s->rows = obj ? s->n + 1 : s->n;
  return BASQ_OK;
}

// the context's device buffer for host-buffer calls and the side stream their copies travel on
static int ensure_host_buffer(basq_ctx* ctx, size_t need) {
  if (need > ctx->host_x_bytes) {
    if (ctx->host_x) {
      BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
      if (ctx->side) BASQ_CUDA(cudaStreamSynchronize(ctx->side));
      BASQ_CUDA(cudaFree(ctx->host_x));
      ctx->host_x = nullptr;
      ctx->host_x_bytes = 0;
    }
    BASQ_CUDA(cudaMalloc(&ctx->host_x, need));
    ctx->host_x_bytes = need;
  }
  return BASQ_OK;
}

static int ensure_side_stream(basq_ctx* ctx) {
  if (!ctx->side) {   // created once per context: stream / event creation and destruction take driver-wide locks
    BASQ_CUDA(cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking));
    BASQ_CUDA(cudaEventCreateWithFlags(&ctx->side_ev[0], cudaEventDisableTiming));
    BASQ_CUDA(cudaEventCreateWithFlags(&ctx->side_ev[1], cudaEventDisableTiming));
  }
  return BASQ_OK;
}

static int recombine_host_impl(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X_host, int64_t N,
                               const void* Z_host, int64_t M, const double* U_host, int q, const double* Omega_host,
                               int niter, const double* mu_host, int64_t* idx_out_host, double* w_out_host,
                               int* n_out_host) {
  BASQ_CHECK(ctx && desc && X_host && Z_host && idx_out_host && w_out_host && n_out_host, BASQ_ERR_INVALID,
             "basq_recombine_host: NULL argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  const size_t esz = desc->dtype == BASQ_F64 ? 8 : 4;
  trace_point(ctx, "host: enter");
  // All call-lifetime device copies of the host arguments live in ONE buffer the context keeps between calls,
  // outside the block cache: the cache then sees exactly the requests of the device-resident path.
  DevBuf dOm;
  Piece dX, dZ, dU, didx, dw;
  double* dmu_p = nullptr;
  {
    auto up = [](size_t b) { return (b + 255) / 256 * 256; };
    const size_t bX = up(esz * (size_t)N * desc->d), bmu = mu_host ? up(sizeof(double) * (size_t)N) : 0;
    const size_t bZ = up(esz * (size_t)M * desc->d), bU = up(sizeof(double) * (size_t)q * M);
    const size_t bi = up(sizeof(int64_t) * (q + 1)), bw = up(sizeof(double) * (q + 1));
    const size_t need = bX + bmu + bZ + bU + bi + bw;
    ctx->staged_N = -1;   // the buffer is about to be overwritten
    BASQ_TRY(ensure_host_buffer(ctx, need));
    unsigned char* base = static_cast<unsigned char*>(ctx->host_x);
    dX.p = base;
    if (mu_host) dmu_p = reinterpret_cast<double*>(base + bX);
    dZ.p = base + bX + bmu;
    dU.p = base + bX + bmu + bZ;
    didx.p = base + bX + bmu + bZ + bU;
    dw.p = base + bX + bmu + bZ + bU + bi;
  }
  // The candidates (the bulk of the bytes) travel on a side stream while the basis is built from the
  // landmarks on the main stream: the Nystrom phase hides the host-to-device copy.
  BASQ_TRY(ensure_side_stream(ctx));
  cudaStream_t side = ctx->side;
  cudaEvent_t x_ready = ctx->side_ev[0], buffers_ready = ctx->side_ev[1];
  auto cleanup = [&]() { cudaStreamSynchronize(side); };   // the next call reuses the candidate buffer: the copy must be over
  // Landmarks and the test matrix go first (the copy engine serves requests in order, and the basis
  // cannot start without them); the candidates follow on the side stream.
  int rc = BASQ_OK;
  {
    cudaError_t e2 = cudaMemcpyAsync(dZ.p, Z_host, esz * (size_t)M * desc->d, cudaMemcpyHostToDevice, ctx->stream);
    if (e2 == cudaSuccess && U_host)
      e2 = cudaMemcpyAsync(dU.p, U_host, sizeof(double) * (size_t)q * M, cudaMemcpyHostToDevice, ctx->stream);
    if (e2 == cudaSuccess && !U_host && Omega_host) {
      rc = dOm.alloc(ctx, sizeof(double) * (size_t)M * q);
      if (rc == BASQ_OK)
        e2 = cudaMemcpyAsync(dOm.p, Omega_host, sizeof(double) * (size_t)M * q, cudaMemcpyHostToDevice, ctx->stream);
    }
    if (e2 != cudaSuccess) {
      set_error("basq_recombine_host: landmark copy failed: %s", cudaGetErrorString(e2));
      rc = BASQ_ERR_CUDA;
    }
  }
  if (rc != BASQ_OK) {
    cleanup();
    return rc;
  }
  BASQ_CUDA(cudaEventRecord(buffers_ready, ctx->stream));        // earlier work on the main stream may still read the candidate buffer
  BASQ_CUDA(cudaStreamWaitEvent(side, buffers_ready, 0));
  cudaError_t ce = cudaMemcpyAsync(dX.p, X_host, esz * (size_t)N * desc->d, cudaMemcpyHostToDevice, side);
  if (ce == cudaSuccess && mu_host)
    ce = cudaMemcpyAsync(dmu_p, mu_host, sizeof(double) * N, cudaMemcpyHostToDevice, side);
  if (ce == cudaSuccess) ce = cudaEventRecord(x_ready, side);
  if (ce != cudaSuccess) {
    cleanup();
    set_error("basq_recombine_host: candidate copy failed: %s", cudaGetErrorString(ce));
    return BASQ_ERR_CUDA;
  }
  if (!U_host) {
    trace_point(ctx, "host: Z / Omega copies issued");
    rc = nystrom_basis(ctx, desc, dZ.p, M, q, Omega_host ? dOm.as<double>() : nullptr, niter, dU.as<double>(), nullptr,
                       nullptr);
  }
  if (rc == BASQ_OK && cudaStreamWaitEvent(ctx->stream, x_ready, 0) != cudaSuccess) rc = BASQ_ERR_CUDA;
  if (rc != BASQ_OK) {
    cleanup();
    return rc;
  }
  trace_point(ctx, "host: inputs + basis on device");
  int n_out = 0;
  rc = recombine_impl(ctx, desc, dX.p, N, dZ.p, M, dU.as<double>(), q, dmu_p,
                      didx.as<int64_t>(), dw.as<double>(), &n_out);
  cleanup();
  if (rc != BASQ_OK) return rc;
  BASQ_CUDA(cudaMemcpyAsync(idx_out_host, didx.p, sizeof(int64_t) * n_out, cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaMemcpyAsync(w_out_host, dw.p, sizeof(double) * n_out, cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  *n_out_host = n_out;
  trace_point(ctx, "host: results copied back");
  return BASQ_OK;
}

int basq_recombine_host(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X_host, int64_t N,
                        const void* Z_host, int64_t M, const double* U_host, int q, const double* Omega_host,
                        int niter, const double* mu_host, int64_t* idx_out_host, double* w_out_host,
                        int* n_out_host) {
  const int rc = recombine_host_impl(ctx, desc, X_host, N, Z_host, M, U_host, q, Omega_host, niter, mu_host,
                                     idx_out_host, w_out_host, n_out_host);
  if (ctx) basq_ctx_trim(ctx, -1);
  return rc;
}

// ---- host buffers for the sharded path -------------------------------------------------------------------
int basq_ctx_stage_candidates(basq_ctx* ctx, const void* X_host, int64_t N_loc, int d, int dtype, const double* mu_host) {
  BASQ_CHECK(ctx && (X_host || N_loc == 0) && N_loc >= 0 && d >= 1 && d <= BASQ_MAX_DIM &&
                 (dtype == BASQ_F32 || dtype == BASQ_F64),
             BASQ_ERR_INVALID, "basq_ctx_stage_candidates: bad argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  const size_t esz = dtype == BASQ_F64 ? 8 : 4;
  auto up = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t bX = up(esz * (size_t)N_loc * d), bmu = mu_host ? up(sizeof(double) * (size_t)N_loc) : 0;
  ctx->staged_N = -1;
  BASQ_TRY(ensure_host_buffer(ctx, std::max<size_t>(bX + bmu, 256)));
  BASQ_TRY(ensure_side_stream(ctx));
  // earlier work on the main stream may still read the buffer (a session under construction)
  BASQ_CUDA(cudaEventRecord(ctx->side_ev[1], ctx->stream));
  BASQ_CUDA(cudaStreamWaitEvent(ctx->side, ctx->side_ev[1], 0));
  unsigned char* base = static_cast<unsigned char*>(ctx->host_x);
  if (N_loc > 0) BASQ_CUDA(cudaMemcpyAsync(base, X_host, esz * (size_t)N_loc * d, cudaMemcpyHostToDevice, ctx->side));
  ctx->staged_mu = nullptr;
  if (mu_host && N_loc > 0) {
    ctx->staged_mu = reinterpret_cast<double*>(base + bX);
    BASQ_CUDA(cudaMemcpyAsync(ctx->staged_mu, mu_host, sizeof(double) * (size_t)N_loc, cudaMemcpyHostToDevice, ctx->side));
  }
  BASQ_CUDA(cudaEventRecord(ctx->side_ev[0], ctx->side));
  ctx->staged_N = N_loc;
  ctx->staged_d = d;
  ctx->staged_dtype = dtype;
  return BASQ_OK;
}

int basq_session_create_staged(basq_ctx* ctx, const basq_kernel_desc* desc, int64_t N_loc, int64_t N_glob, int64_t idx_base,
                               const void* Z, int64_t M, const double* U, int q, basq_session** out) {
  BASQ_CHECK(ctx && desc && out, BASQ_ERR_INVALID, "basq_session_create_staged: NULL argument");
  *out = nullptr;
  BASQ_CHECK(ctx->staged_N == N_loc && ctx->staged_d == desc->d && ctx->staged_dtype == desc->dtype, BASQ_ERR_INVALID,
             "basq_session_create_staged: the staged candidates (%lld x %d, dtype %d) do not match the call (%lld x %d, dtype %d)",
             (long long)ctx->staged_N, ctx->staged_d, ctx->staged_dtype, (long long)N_loc, desc->d, desc->dtype);
  BASQ_CUDA(cudaSetDevice(ctx->device));
  BASQ_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->side_ev[0], 0));
  std::unique_ptr<basq_session> s(new (std::nothrow) basq_session());
  BASQ_CHECK(s, BASQ_ERR_INVALID, "out of host memory");
  BASQ_TRY(session_create_impl(ctx, desc, N_loc > 0 ? ctx->host_x : nullptr, N_loc, N_glob, idx_base, Z, M, U, q,
                               ctx->staged_mu, 0, s.get()));
  *out = s.release();
  return BASQ_OK;
}

int basq_session_create(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N_loc, int64_t N_glob,
                        int64_t idx_base, const void* Z, int64_t M, const double* U, int q, const double* mu,
                        basq_session** out) {
  BASQ_CHECK(ctx && out, BASQ_ERR_INVALID, "basq_session_create: NULL argument");
  *out = nullptr;
  BASQ_CUDA(cudaSetDevice(ctx->device));
  std::unique_ptr<basq_session> s(new (std::nothrow) basq_session());
  BASQ_CHECK(s, BASQ_ERR_INVALID, "out of host memory");
  BASQ_TRY(session_create_impl(ctx, desc, X, N_loc, N_glob, idx_base, Z, M, U, q, mu, 0, s.get()));
  *out = s.release();
  return BASQ_OK;
}

void basq_session_destroy(basq_session* s) {
  if (!s) return;
  basq_ctx* ctx = s->ctx;
  delete s;
  if (ctx) basq_ctx_trim(ctx, -1);
}

int basq_session_count(const basq_session* s, int64_t* R_loc_host) {
  BASQ_CHECK(s && R_loc_host, BASQ_ERR_INVALID, "NULL argument");
  *R_loc_host = s->pool.count;
  return BASQ_OK;
}

int basq_session_partial(basq_session* s, int64_t R_glob, int64_t off_glob, double* A_out) {
  BASQ_CHECK(s && A_out, BASQ_ERR_INVALID, "NULL argument");
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  BASQ_TRY(session_pass_begin(s, R_glob, off_glob, 1));
  LevelTree tree;
  tree.begin(s->S, 1, R_glob);
  return session_level(s, 0, (int)tree.node.size(), tree.node.data(), tree.ppos.data(), tree.fpar.data(), A_out);
}

int basq_session_cell_factor(const basq_session* s, int64_t R_glob, int64_t R_loc_max, int* F_out_host) {
  BASQ_CHECK(s && F_out_host, BASQ_ERR_INVALID, "NULL argument");
  *F_out_host = choose_cell_factor(s, R_glob, R_loc_max);
  return BASQ_OK;
}

int basq_session_pass_begin(basq_session* s, int64_t R_glob, int64_t off_glob, int F) {
  BASQ_CHECK(s, BASQ_ERR_INVALID, "NULL argument");
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  return session_pass_begin(s, R_glob, off_glob, F);
}

int basq_session_landmarks(const basq_session* s, int* Mtot_out_host) {
  BASQ_CHECK(s && Mtot_out_host, BASQ_ERR_INVALID, "NULL argument");
  *Mtot_out_host = s->Mtot;
  return BASQ_OK;
}

int basq_session_level_fold(basq_session* s, int lvl, int K, const int* node_host, double* Gf_out, int64_t ld_gf) {
  BASQ_CHECK(s && node_host && Gf_out && ld_gf >= K, BASQ_ERR_INVALID, "basq_session_level_fold: bad argument");
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  return session_level_fold(s, lvl, K, node_host, Gf_out, ld_gf);
}

int basq_session_level_project(basq_session* s, int lvl, int K, const int* node_host, const int* ppos_host,
                               const double* fpar_host, const double* Gf_rows, int64_t ld_gf, int row0, int nrows,
                               double* A_out) {
  BASQ_CHECK(s && node_host && fpar_host && A_out && (lvl == 0 || ppos_host) && (Gf_rows || nrows == 0) && ld_gf >= K,
             BASQ_ERR_INVALID, "basq_session_level_project: bad argument");
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  return session_level_project(s, lvl, K, node_host, ppos_host, fpar_host, Gf_rows, ld_gf, row0, nrows, A_out);
}

int basq_session_level(basq_session* s, int lvl, int K, const int* node_host, const int* ppos_host,
                       const double* fpar_host, double* A_out) {
  BASQ_CHECK(s && node_host && fpar_host && A_out && (lvl == 0 || ppos_host), BASQ_ERR_INVALID, "NULL argument");
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  return session_level(s, lvl, K, node_host, ppos_host, fpar_host, A_out);
}

int basq_session_reproducible(const basq_session* s, int* on_host) {
  BASQ_CHECK(s && on_host, BASQ_ERR_INVALID, "NULL argument");
  *on_host = s->repro ? 1 : 0;
  return BASQ_OK;
}

int basq_session_grid_maxima(basq_session* s, double* max_host) {
  BASQ_CHECK(s && max_host, BASQ_ERR_INVALID, "NULL argument");
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  return session_grid_local(s, max_host);
}

int basq_session_set_grid(basq_session* s, int64_t R_glob, const double* max_host) {
  BASQ_CHECK(s && max_host, BASQ_ERR_INVALID, "NULL argument");
  return session_set_grid(s, R_glob, max_host);
}

int basq_session_level_fold_exact(basq_session* s, int lvl, int K, const int* node_host, double* Gf_out,
                                  int64_t ld_gf) {
  BASQ_CHECK(s && node_host && Gf_out && ld_gf >= K, BASQ_ERR_INVALID, "basq_session_level_fold_exact: bad argument");
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  return session_level_fold_exact(s, lvl, K, node_host, Gf_out, ld_gf);
}

int basq_session_level_project_exact(basq_session* s, int lvl, int K, const int* node_host, const int* ppos_host,
                                     const double* fpar_host, const double* Gf, int64_t ld_gf, double* A_out) {
  BASQ_CHECK(s && node_host && fpar_host && A_out && Gf && (lvl == 0 || ppos_host) && ld_gf >= K, BASQ_ERR_INVALID,
             "basq_session_level_project_exact: bad argument");
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  return session_level_project_exact(s, lvl, K, node_host, ppos_host, fpar_host, Gf, ld_gf, A_out);
}

int basq_session_apply(basq_session* s, int64_t R_glob, int64_t off_glob, const double* omega,
                       int64_t* R_loc_new_host) {
  BASQ_CHECK(s && omega, BASQ_ERR_INVALID, "NULL argument");
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  std::vector<double> h((size_t)s->S);
  BASQ_CUDA(cudaMemcpyAsync(h.data(), omega, sizeof(double) * s->S, cudaMemcpyDeviceToHost, s->ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(s->ctx->stream));
  return session_apply_impl(s, R_glob, off_glob, 1, h.data(), R_loc_new_host);
}

int basq_session_apply_cells(basq_session* s, int64_t R_glob, int64_t off_glob, int F, const double* factor_host,
                             int64_t* R_loc_new_host) {
  BASQ_CHECK(s && factor_host, BASQ_ERR_INVALID, "NULL argument");
  BASQ_CHECK(F >= 1 && F <= BASQ_MAX_CELL_FACTOR && (F & (F - 1)) == 0, BASQ_ERR_INVALID, "apply: bad cell factor %d", F);
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  return session_apply_impl(s, R_glob, off_glob, F, factor_host, R_loc_new_host);
}

int basq_session_result(basq_session* s, int64_t* idx_out, double* w_out, int cap, int* n_out_host) {
  BASQ_CHECK(s && idx_out && w_out && n_out_host, BASQ_ERR_INVALID, "NULL argument");
  BASQ_CHECK(s->pool.count <= cap, BASQ_ERR_INVALID, "result: %lld live points exceed capacity %d",
             (long long)s->pool.count, cap);
  BASQ_CUDA(cudaSetDevice(s->ctx->device));
  BASQ_TRY(extract_result(s->ctx, s->pool, s->idx_base, idx_out, w_out));
  BASQ_CUDA(cudaStreamSynchronize(s->ctx->stream));
  *n_out_host = (int)s->pool.count;
  return BASQ_OK;
}

}  // extern "C"
