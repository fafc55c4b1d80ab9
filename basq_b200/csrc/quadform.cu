// Weighted kernel double sums over point sets, without forming the Gram matrix:
//   basq_kernel_quadform  Q(X, a)       = a^T basq_gram(desc, X, X) a        (diagonal terms included)
//   basq_kernel_bilinear  B(X, a; Y, b) = sum_ij a_i b_j kernel(x_i, y_j)     (the kernel function alone)
// Q is SOBER's full_quadrature variance w^T K(X, X) w (SOBER/BASQ/_basq.py:48-81) at candidate scale, and
// the squared worst-case error of a quadrature rule, Q(X, mu - w~) (gp.worst_case_error).
//
// The N-scale work runs on the set-sum kernels (setsum.cu) with the roles of landmark_dot_tc (gram.cu):
// a block of L rows of X is prepared as landmarks, the weighted points are the records, and every
// landmark gets 8 partial sums (one per record set).  For Q the block meets the records from its own
// first row onward: its own records once, the later ones twice (symmetry), so about N^2 / 2 + N L / 2
// pairs are evaluated.  The records are built without the zero-weight filter (factor = weight): record
// p is row p, so a block's landmarks and its records line up without a gather.
//
// Posterior-covariance modes are linear in k and separate (DESIGN.md, "Weighted double sums"):
//   a^T C b = a~^T K b~ - (K_{Xobs,X} a~)^T W (K_{Xobs,Y} b~),   a~ = a (PRED_COV), a (.) m(x) (WSABI-L);
// the two n_obs-vectors are one more set sum each, with the observations as landmarks.  WSABI-M and MMLT
// need C per pair: every block gets Az = K(X_B, Xobs) W and its per-point factors as landmark factors
// (posterior_az / nl_sweep_prepare, shared with the sessions) and runs the non-linear set sums (nlsum.cuh
// for fp32, the chunked fp64-GEMM correction otherwise).  fp32 calls in these modes compute
// kappa = max_i |Az_i|_1 over all rows before the sweep and are promoted to fp64 beyond kappa_max.
//
// Every sum is deterministic: per-block partials in a fixed order, then one fixed-order sum; no atomics.
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace basq {

namespace {

constexpr int QF_SETS = 8;                   // partial sums per landmark: 8 sets fill the set-sum tiles
constexpr int QF_THREADS = 256;
constexpr int QF_ROWS = 16 * QF_THREADS;     // rows per reduction block (one partial each)

// sum of every thread's v over the block, pairwise in a fixed tree (same bits from run to run)
__device__ double qf_block_sum(double v) {
  __shared__ double sh[QF_THREADS];
  sh[threadIdx.x] = v;
  __syncthreads();
  for (int w = QF_THREADS / 2; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  return sh[0];
}

// parts[block] = scale * sum over the block's rows m of c[m] * sum_{j < cols} G[m, j]
__global__ void __launch_bounds__(QF_THREADS) qf_reduce_kernel(const double* __restrict__ G, int64_t rows, int cols,
                                                               const double* __restrict__ c, double scale,
                                                               double* __restrict__ parts) {
  const int64_t r0 = (int64_t)blockIdx.x * QF_ROWS;
  const int64_t r1 = min(rows, r0 + QF_ROWS);
  double s = 0.0;
  for (int64_t m = r0 + threadIdx.x; m < r1; m += QF_THREADS) {
    const double* g = G + m * cols;
    double row = 0.0;
    for (int j = 0; j < cols; ++j) row += g[j];
    s = fma(c[m], row, s);
  }
  const double t = qf_block_sum(s);
  if (threadIdx.x == 0) parts[blockIdx.x] = scale * t;
}

// Diagonal terms of basq_gram(X, X) that the kernel function lacks, a_i^2 (kappa^_ii - kappa_ii): the
// likelihood noise s2 enters the covariance C_ii before the warping, the jitter after it.
//   linear modes: s2 f_i^2 (f = m(x) for WSABI-L, 1 otherwise)
//   WSABI-M:      f C f + C^2 / 2  ->  s2 f_i^2 + s2 C_ii + s2^2 / 2
//   MMLT:         f^2 expm1(C)     ->  f_i^2 exp(C_ii) expm1(s2)
__global__ void __launch_bounds__(QF_THREADS) qf_diag_kernel(const double* __restrict__ a, const double* __restrict__ f,
                                                             const double* __restrict__ C, int64_t n, int mode,
                                                             double s2, double diag_add, double* __restrict__ parts) {
  const int64_t r0 = (int64_t)blockIdx.x * QF_ROWS;
  const int64_t r1 = min(n, r0 + QF_ROWS);
  double s = 0.0;
  for (int64_t i = r0 + threadIdx.x; i < r1; i += QF_THREADS) {
    const double fi = f ? f[i] : 1.0;
    double dk;
    if (mode == BASQ_WSABI_M) dk = s2 * fi * fi + s2 * C[i] + 0.5 * s2 * s2;
    else if (mode == BASQ_MMLT_G) dk = fi * fi * exp(C[i]) * expm1(s2);
    else dk = s2 * fi * fi;
    s = fma(a[i] * a[i], dk + diag_add, s);
  }
  const double t = qf_block_sum(s);
  if (threadIdx.x == 0) parts[blockIdx.x] = t;
}

// *out = sum of parts[0 .. n) in a fixed order (one block)
__global__ void __launch_bounds__(QF_THREADS) qf_sum_kernel(const double* __restrict__ parts, int n,
                                                            double* __restrict__ out) {
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += QF_THREADS) s += parts[i];
  const double t = qf_block_sum(s);
  if (threadIdx.x == 0) *out = t;
}

// out[i] = w[i] * f[i] (f may be NULL: out = w); *bad = 1 if a weight is not finite
__global__ void qf_weights_kernel(const double* __restrict__ w, const double* __restrict__ f, int64_t n,
                                  double* __restrict__ out, int* __restrict__ bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double v = w[i];
  if (!isfinite(v)) atomicOr(bad, 1);   // integer flag: the order of the writes does not matter
  out[i] = f ? v * f[i] : v;
}

// measure weight of record p = w[p] (the non-linear set sums weigh nl(C) by it; wf holds the factor)
__global__ void qf_record_weight_kernel(unsigned char* __restrict__ recs, int rec_bytes, int64_t n,
                                        const double* __restrict__ w) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) reinterpret_cast<double*>(recs + p * rec_bytes)[1] = w[p];
}

// C_ii = var_i - s2: the posterior variance without the likelihood noise
__global__ void qf_cov_diag_kernel(double* __restrict__ var, int64_t n, double s2) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) var[i] -= s2;
}

// per-block partials, summed once at the end
struct Partials {
  DevBuf buf;
  int n = 0, cap = 0;
  int reserve(basq_ctx* ctx, int c) {
    cap = c;
    return buf.alloc(ctx, sizeof(double) * (size_t)(c + 1));
  }
  double* take(int k) {
    double* p = buf.as<double>() + n;
    n += k;
    return p;
  }
};

int reduce_rows(basq_ctx* ctx, Partials* parts, const double* G, int64_t rows, int cols, const double* coef,
                double scale) {
  const int nb = ceil_div(rows, QF_ROWS);
  BASQ_CHECK(parts->n + nb <= parts->cap, BASQ_ERR_INVALID, "quadform: partial-sum buffer too small");
  qf_reduce_kernel<<<nb, QF_THREADS, 0, ctx->stream>>>(G, rows, cols, coef, scale, parts->take(nb));
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

// One operand of a form: the points, the landmark coefficients wt (weights, times m(x) for WSABI-L), the
// per-point factor of the warped modes, and the records.
struct Operand {
  const void* X = nullptr;
  int64_t n = 0;
  const double* w = nullptr;
  DevBuf wt, fac;
  RecPool pool;
};

int prepare_operand(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const LmView& lmobs,
                    Operand* op, bool records) {
  const int mode = desc->mode;
  const bool nonlin = mode == BASQ_WSABI_M || mode == BASQ_MMLT_G;
  if (mode == BASQ_WSABI_L || nonlin) {
    BASQ_TRY(op->fac.alloc(ctx, sizeof(double) * op->n));
    BASQ_TRY(warp_factor(ctx, desc, kp, lmobs, op->X, op->n, op->fac.as<double>()));
  }
  DevBuf bad;
  BASQ_TRY(bad.alloc(ctx, sizeof(int)));
  BASQ_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), ctx->stream));
  BASQ_TRY(op->wt.alloc(ctx, sizeof(double) * op->n));
  qf_weights_kernel<<<(unsigned)ceil_div64(op->n, 256), 256, 0, ctx->stream>>>(
      op->w, mode == BASQ_WSABI_L ? op->fac.as<double>() : nullptr, op->n, op->wt.as<double>(), bad.as<int>());
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  int bad_host = 0;
  BASQ_CUDA(cudaMemcpyAsync(&bad_host, bad.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  BASQ_CHECK(!bad_host, BASQ_ERR_NUMERIC, "quadform: the weights contain a non-finite value");
  if (!records) return BASQ_OK;
  // uniform weight 1 keeps every point (record p = row p); one buffer, no recombination rounds
  if (!nonlin)
    return build_records(ctx, kp, desc->dtype, op->X, op->n, 1.0, nullptr, op->wt.as<double>(), true, &op->pool, false);
  BASQ_TRY(build_records(ctx, kp, desc->dtype, op->X, op->n, 1.0, nullptr, op->fac.as<double>(), false, &op->pool, false));
  qf_record_weight_kernel<<<(unsigned)ceil_div64(op->n, 256), 256, 0, ctx->stream>>>(
      op->pool.buf[0].as<unsigned char>(), op->pool.rec_bytes, op->n, op->w);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

SetSumArgs sweep_args(const RecPool& pool, const LmView& lm, int nl, const double* sz, double* G) {
  SetSumArgs s;
  s.pool = &pool;
  s.lm = lm;
  s.off_glob = 0;
  s.S = QF_SETS;
  s.p_lo = s.p_hi = 0;
  s.nl = nl;
  s.corrT = nullptr;
  s.ld_corr = 0;
  s.sz = sz;
  s.G = G;
  s.ldg = QF_SETS;
  s.accumulate = false;
  return s;
}

// G[:, 0..QF_SETS) = set sums of records [p_lo, p_hi) against lm (linear modes)
int sweep(basq_ctx* ctx, const KParams& kp, const LmView& lm, const RecPool& pool, int64_t p_lo, int64_t p_hi,
          double* G) {
  BASQ_CUDA(cudaMemsetAsync(G, 0, sizeof(double) * (size_t)lm.count * QF_SETS, ctx->stream));
  if (p_hi <= p_lo) return BASQ_OK;
  SetSumArgs s = sweep_args(pool, lm, NL_LIN, nullptr, G);
  s.p_lo = p_lo;
  s.p_hi = p_hi;
  s.accumulate = true;
  return set_sums(ctx, kp, s);
}

// u[o] = sum_p wt_p k(xobs_o, x_p) over all records of op
int obs_sums(basq_ctx* ctx, const KParams& kp, const LmView& lmobs, const Operand& op, double* u) {
  const int n_obs = lmobs.count;
  DevBuf G;
  BASQ_TRY(G.alloc(ctx, sizeof(double) * (size_t)n_obs * QF_SETS));
  BASQ_TRY(sweep(ctx, kp, lmobs, op.pool, 0, op.pool.count, G.as<double>()));
  BASQ_TRY(rowsum_cols(ctx, G.as<double>(), n_obs, QF_SETS, 0.0, u));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));   // G goes out of scope
  return BASQ_OK;
}

// landmark rows per block: one work item of the set-sum kernel is 256 landmarks x 8 sets
int64_t block_rows(basq_ctx* ctx, int64_t N) { return std::min<int64_t>(N, (int64_t)std::max(ctx->num_sms, 1) * 256); }

// kappa = max_i |(K(X, Xobs) W)_i|_1 over every row of X, block by block
int all_rows_kappa(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const void* X, int64_t N,
                   double* kappa) {
  const int64_t L = block_rows(ctx, N);
  const size_t esz = desc->dtype == BASQ_F32 ? 4 : 8;
  DevBuf Az;
  BASQ_TRY(Az.alloc(ctx, sizeof(double) * (size_t)L * desc->n_obs));
  Landmarks lm;
  *kappa = 0.0;
  for (int64_t r0 = 0; r0 < N; r0 += L) {
    const int64_t cnt = std::min(N, r0 + L) - r0;
    BASQ_TRY(prep_landmarks(ctx, kp, desc->dtype, (const unsigned char*)X + (size_t)r0 * desc->d * esz, cnt, nullptr,
                            0, &lm));
    double k = 0.0;
    BASQ_TRY(posterior_az(ctx, desc, kp, lm.view(), Az.as<double>(), &k));
    *kappa = std::max(*kappa, k);
  }
  ctx->last_kappa = *kappa;
  return BASQ_OK;
}

// sym: Q(X, a) (Y, b ignored); else B(X, a; Y, b)
int form_impl(basq_ctx* ctx, const basq_kernel_desc* desc_in, const void* X, int64_t N, const double* a,
              const void* Y, int64_t Mb, const double* b, bool sym, double* out_host) {
  const char* who = sym ? "basq_kernel_quadform" : "basq_kernel_bilinear";
  BASQ_CHECK(ctx && desc_in && X && a && out_host && (sym || (Y && b)), BASQ_ERR_INVALID, "%s: NULL argument", who);
  BASQ_CHECK(N >= 1 && (sym || Mb >= 1), BASQ_ERR_INVALID, "%s: empty operand", who);
  const int64_t lim = (1ll << 31) - 1024;
  BASQ_CHECK(N < lim && (sym || Mb < lim), BASQ_ERR_UNSUPPORTED, "%s: at most 2^31 - 1024 points per operand", who);
  const int mode = desc_in->mode;
  BASQ_CHECK(mode >= BASQ_PLAIN && mode <= BASQ_MMLT_G, BASQ_ERR_INVALID, "%s: unknown mode %d", who, mode);
  BASQ_CHECK(mode == BASQ_PLAIN || (desc_in->n_obs > 0 && desc_in->Xobs && desc_in->W && desc_in->alpha),
             BASQ_ERR_INVALID, "%s: posterior kernels need the GP caches (n_obs, Xobs, W, alpha)", who);
  BASQ_CUDA(cudaSetDevice(ctx->device));
  if (sym) { Y = X; Mb = N; b = a; }
  const bool nonlin = mode == BASQ_WSABI_M || mode == BASQ_MMLT_G;

  EvalRoute route;
  BASQ_TRY(route.begin(ctx, desc_in, X, N, Y, Mb));
  const basq_kernel_desc* desc = &route.desc;
  KParams kp;
  BASQ_TRY(make_kparams(desc, &kp));
  BASQ_TRY(compute_center(ctx, desc, route.pts[0], N, &kp));
  if (nonlin && route.can_promote(ctx)) {
    // conditioning guard, over every landmark row before the sweep (as sessions do for Z)
    double kappa = 0.0;
    BASQ_TRY(all_rows_kappa(ctx, desc, kp, route.pts[0], N, &kappa));
    if (kappa > ctx->kappa_max) {
      BASQ_TRY(route.promote(ctx));
      BASQ_TRY(make_kparams(desc, &kp));
      BASQ_TRY(compute_center(ctx, desc, route.pts[0], N, &kp));
    }
  }
  const void* Xe = route.pts[0];
  const void* Ye = route.pts[1];
  const size_t esz = desc->dtype == BASQ_F32 ? 4 : 8;

  Landmarks lmobs;
  if (mode != BASQ_PLAIN) BASQ_TRY(prep_landmarks(ctx, kp, desc->dtype, desc->Xobs, desc->n_obs, nullptr, 0, &lmobs));

  Operand opx, opy;
  opx.X = Xe; opx.n = N; opx.w = a;
  opy.X = Ye; opy.n = Mb; opy.w = b;
  // the X operand needs records for the linear posterior correction (and for Q, where it is both operands)
  BASQ_TRY(prepare_operand(ctx, desc, kp, lmobs.view(), &opx, sym || (mode != BASQ_PLAIN && !nonlin)));
  if (!sym) BASQ_TRY(prepare_operand(ctx, desc, kp, lmobs.view(), &opy, true));
  const Operand& rec = sym ? opx : opy;

  const int64_t L = block_rows(ctx, N);
  const int64_t nblk = ceil_div64(N, L);
  Partials parts;
  BASQ_TRY(parts.reserve(ctx, (int)(2 * nblk * ceil_div(L, QF_ROWS) + ceil_div(N, QF_ROWS) +
                                     ceil_div(std::max(desc->n_obs, 1), QF_ROWS))));
  // own: the block's own records (Q) or all records (B), once; later: the rows after the block (Q), twice
  DevBuf Gown, Glater, Az;
  BASQ_TRY(Gown.alloc(ctx, sizeof(double) * (size_t)L * QF_SETS));
  if (sym) BASQ_TRY(Glater.alloc(ctx, sizeof(double) * (size_t)L * QF_SETS));
  if (nonlin) BASQ_TRY(Az.alloc(ctx, sizeof(double) * (size_t)L * desc->n_obs));
  const int nl = mode == BASQ_WSABI_M ? NL_WSABIM : (mode == BASQ_MMLT_G ? NL_MMLT : NL_LIN);
  {
    PhaseTimer timer(ctx, PH_SETSUM);
    Landmarks lm;
    double kappa = 0.0;
    for (int64_t r0 = 0; r0 < N; r0 += L) {
      const int64_t r1 = std::min(N, r0 + L), cnt = r1 - r0;
      BASQ_TRY(prep_landmarks(ctx, kp, desc->dtype, (const unsigned char*)Xe + (size_t)r0 * desc->d * esz, cnt, nullptr,
                              0, &lm));
      const int64_t own_lo = sym ? r0 : 0, own_hi = sym ? r1 : Mb;
      if (!nonlin) {
        BASQ_TRY(sweep(ctx, kp, lm.view(), rec.pool, own_lo, own_hi, Gown.as<double>()));
        if (sym) BASQ_TRY(sweep(ctx, kp, lm.view(), rec.pool, r1, N, Glater.as<double>()));
      } else {
        // the block's landmark side: Az and the factors of its rows (as a session prepares Z)
        double k = 0.0;
        BASQ_TRY(posterior_az(ctx, desc, kp, lm.view(), Az.as<double>(), &k));
        kappa = std::max(kappa, k);
        const double* sz = opx.fac.as<double>() + r0;
        NlSweep w;
        BASQ_TRY(nl_sweep_prepare(ctx, desc, kp, Az.as<double>(), (int)cnt, sz, rec.n, &w));
        SetSumArgs s = sweep_args(rec.pool, lm.view(), nl, sz, Gown.as<double>());
        BASQ_TRY(nl_sweep_sums(ctx, kp, nl, &w, rec.pool, lm.view(), lmobs.view(), 0, QF_SETS, own_lo, own_hi,
                               Gown.as<double>(), QF_SETS, &s));
        if (sym) {
          s = sweep_args(rec.pool, lm.view(), nl, sz, Glater.as<double>());
          BASQ_TRY(nl_sweep_sums(ctx, kp, nl, &w, rec.pool, lm.view(), lmobs.view(), 0, QF_SETS, r1, N,
                                 Glater.as<double>(), QF_SETS, &s));
        }
        BASQ_CUDA(cudaStreamSynchronize(ctx->stream));   // w's buffers go out of scope
      }
      BASQ_TRY(reduce_rows(ctx, &parts, Gown.as<double>(), cnt, QF_SETS, opx.wt.as<double>() + r0, 1.0));
      if (sym) BASQ_TRY(reduce_rows(ctx, &parts, Glater.as<double>(), cnt, QF_SETS, opx.wt.as<double>() + r0, 2.0));
    }
    if (nonlin) ctx->last_kappa = kappa;
  }

  DevBuf u, v, t;
  if (mode != BASQ_PLAIN && !nonlin) {
    // - (K_{Xobs,X} a~)^T W (K_{Xobs,Y} b~)
    PhaseTimer timer(ctx, PH_GP);
    const int n_obs = desc->n_obs;
    BASQ_TRY(u.alloc(ctx, sizeof(double) * n_obs));
    BASQ_TRY(t.alloc(ctx, sizeof(double) * n_obs));
    BASQ_TRY(obs_sums(ctx, kp, lmobs.view(), opx, u.as<double>()));
    const double* vv = u.as<double>();
    if (!sym) {
      BASQ_TRY(v.alloc(ctx, sizeof(double) * n_obs));
      BASQ_TRY(obs_sums(ctx, kp, lmobs.view(), opy, v.as<double>()));
      vv = v.as<double>();
    }
    BASQ_TRY(dgemm(ctx, false, false, n_obs, 1, n_obs, 1.0, desc->W, n_obs, vv, 1, 0.0, t.as<double>(), 1));
    BASQ_TRY(reduce_rows(ctx, &parts, t.as<double>(), n_obs, 1, u.as<double>(), -1.0));
  }

  DevBuf cdiag;
  if (sym) {
    const double s2 = (mode != BASQ_PLAIN && desc->noise_diag) ? desc->noise : 0.0;
    if (s2 != 0.0 || desc->diag_add != 0.0) {
      if (nonlin) {
        // C_ii from the posterior variance (which includes the likelihood noise)
        BASQ_TRY(cdiag.alloc(ctx, sizeof(double) * N));
        BASQ_TRY(gp_predict_impl(ctx, desc, kp, lmobs.view(), Xe, N, nullptr, cdiag.as<double>()));
        qf_cov_diag_kernel<<<(unsigned)ceil_div64(N, 256), 256, 0, ctx->stream>>>(cdiag.as<double>(), N, desc->noise);
        ctx->launches++;
        BASQ_CUDA(cudaGetLastError());
      }
      const int nb = ceil_div(N, QF_ROWS);
      qf_diag_kernel<<<nb, QF_THREADS, 0, ctx->stream>>>(a, opx.fac.as<double>(), cdiag.as<double>(), N, mode, s2,
                                                          desc->diag_add, parts.take(nb));
      ctx->launches++;
      BASQ_CUDA(cudaGetLastError());
    }
  }

  double* total = parts.buf.as<double>() + parts.cap;
  qf_sum_kernel<<<1, QF_THREADS, 0, ctx->stream>>>(parts.buf.as<double>(), parts.n, total);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  BASQ_CUDA(cudaMemcpyAsync(out_host, total, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

}  // namespace
}  // namespace basq

extern "C" {

int basq_kernel_quadform(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N, const double* a,
                         double* out_host) {
  const int rc = basq::form_impl(ctx, desc, X, N, a, nullptr, 0, nullptr, true, out_host);
  if (ctx) basq_ctx_trim(ctx, -1);
  return rc;
}

int basq_kernel_bilinear(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N, const double* a,
                         const void* Y, int64_t Mb, const double* b, double* out_host) {
  const int rc = basq::form_impl(ctx, desc, X, N, a, Y, Mb, b, false, out_host);
  if (ctx) basq_ctx_trim(ctx, -1);
  return rc;
}

}  // extern "C"
