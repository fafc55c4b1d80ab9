/*
 * basq_b200 - C ABI of the B200-native kernel-recombination (RCHQ) hot path of BASQ.
 *
 * This is the drop-in boundary (SURVEY.md 8b): plain pointers and sizes, no torch types.
 * The reference is pure Python, so there is no existing FFI; each entry point cites the
 * reference function (file:line under the ma921/BASQ tree) whose work it replaces.  The
 * Python shim that a maintainer binds against these symbols is basq_b200/_lib.py (ctypes);
 * INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - every pointer is DEVICE memory on the context's device unless its name ends in _host;
 *   - matrices are dense row-major; coordinates X/Z/Xobs are [rows, d] in desc->dtype;
 *   - all calls are ordered on the context's stream; calls that return host scalars
 *     synchronise that stream before returning;
 *   - return value: BASQ_OK or an error code, text via basq_last_error() (thread local).
 * There is no CPU fallback: without a CUDA device every compute call fails with BASQ_ERR_CUDA.
 */
#ifndef BASQ_B200_H
#define BASQ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BASQ_ABI_VERSION 2
#define BASQ_MAX_DIM 32
#define BASQ_MAX_CELL_FACTOR 16 /* cells per set in a refined pass (basq_session_pass_begin) */

enum basq_status {
  BASQ_OK = 0,
  BASQ_ERR_INVALID = 1,     /* bad argument */
  BASQ_ERR_CUDA = 2,        /* CUDA runtime error / no device */
  BASQ_ERR_NUMERIC = 3,     /* degenerate numerical state (e.g. barrier watchdog, NaN input) */
  BASQ_ERR_UNSUPPORTED = 4  /* shape or option outside the compiled range */
};

enum basq_family { BASQ_RBF = 0, BASQ_MATERN15 = 1, BASQ_MATERN25 = 2 };

/* Kernel handed to recombination (SURVEY.md 8a rows a6-a11). */
enum basq_mode {
  BASQ_PLAIN = 0,     /* covar_module.forward                (SOBER/_kernel.py:27-28)            */
  BASQ_PRED_COV = 1,  /* predictive_covariance               (BASQ/_gp.py:259-277)               */
  BASQ_WSABI_L = 2,   /* m(x) C(x,y) m(y)                    (BASQ/_wsabi.py:205-226, SOBER/_kernel.py:33-47) */
  BASQ_WSABI_M = 3,   /* m(x) C m(y) + C^2/2                 (BASQ/_wsabi.py:228-249)            */
  BASQ_MMLT_G = 4     /* mu_g(x) mu_g(y) (exp C_h - 1)       (SOBER/BASQ/_scale_mmlt.py:258-278) */
};

enum basq_dtype { BASQ_F32 = 0, BASQ_F64 = 1 };

typedef struct basq_ctx basq_ctx;
typedef struct basq_session basq_session;

/* POD description of the GP kernel; extracted from the reference's kernel objects by the shim. */
typedef struct basq_kernel_desc {
  int32_t family;                    /* basq_family */
  int32_t mode;                      /* basq_mode */
  int32_t dtype;                     /* basq_dtype of X / Z / Xobs and of the kernel evaluation */
  int32_t d;                         /* input dimension, 1..BASQ_MAX_DIM */
  double outputscale;                /* ScaleKernel.outputscale (sigma_f^2) */
  double lengthscale[BASQ_MAX_DIM];  /* per-dimension lengthscale (replicate a scalar) */
  double noise;                      /* likelihood.noise (sigma_n^2) */
  double mean_const;                 /* ConstantMean constant (0 for ZeroMean) */
  double diag_add;                   /* jitter added to the first min(a,b) diagonal entries of basq_gram's
                                        result AFTER the warping (BASQ/_wsabi.py:222-224); 0 = off */
  int32_t n_obs;                     /* GP observations; 0 for BASQ_PLAIN */
  int32_t noise_diag;                /* != 0: basq_gram adds `noise` to the first min(a,b) diagonal entries of
                                        the posterior covariance BEFORE any warping - the "+ lik_var" of
                                        BASQ/_gp.py:275-276 (SOBER/_gp.py:297-304 dropped it) */
  const void* Xobs;                  /* [n_obs, d] in dtype */
  const double* W;                   /* [n_obs, n_obs] (K_XX + sigma_n^2 I)^-1, fp64 (BASQ/_gp.py:233-256) */
  const double* alpha;               /* [n_obs] mean cache (K_XX + sigma_n^2 I)^-1 (y - c), fp64 */
  const double* Xobs_f64;            /* optional (may be NULL): the observations in fp64, [n_obs, d].  Used when a
                                        call with fp32 inputs is promoted to the fp64 path (basq_ctx_conditioning):
                                        W belongs to these coordinates, not to their fp32 roundings */
} basq_kernel_desc;

/* ---- context ------------------------------------------------------------------------------ */
int basq_abi_version(void);
const char* basq_last_error(void);
/* stream: a cudaStream_t (0 = the legacy default stream). */
int basq_ctx_create(int device, void* stream, basq_ctx** out);
void basq_ctx_destroy(basq_ctx* ctx);
/* Scratch memory: every ctx owns a private cache of device blocks (plain cudaMalloc blocks, reused whole per
   size class on the context's stream; no CUDA memory pool is involved), so that neither the pass loop nor
   the next call reaches the driver (a 1e7-candidate call holds 7-10 GB).  basq_ctx_trim(ctx, keep_bytes)
   hands the cache back to the driver down to keep_bytes (0: everything, including the candidate buffer of
   basq_recombine_host) - call it when other CUDA code in the process needs the memory, e.g. between the
   BASQ iteration and the GP refit.  keep_bytes < 0 applies the context's automatic keep size, which every
   top-level call also applies before it returns; it is unlimited (no automatic trim) unless the environment
   sets BASQ_POOL_KEEP_MB - a trim is followed by re-allocation at driver speed.  basq_ctx_destroy releases
   everything. */
int basq_ctx_trim(basq_ctx* ctx, int64_t keep_bytes);
/* Scratch memory of the context: bytes cached for reuse (free list of the block cache plus the candidate
   buffer of basq_recombine_host), bytes currently handed out (live sessions), and how many times the cache
   had to go to the driver (cudaMalloc) so far - constant in steady state.  Outputs may be NULL. */
int basq_ctx_memory(const basq_ctx* ctx, uint64_t* cached_bytes_host, uint64_t* live_bytes_host,
                    int64_t* driver_allocs_host);
/* Conditioning guard of the fp32 path.  A posterior-covariance kernel evaluates
   C(z, x) = k(z, x) - (K_ZX W) k(Xobs, x): an evaluation error eps of the kernel values (fp32: ~2e-7
   relative) reaches C as eps * |(K_ZX W)_m|_1 * outputscale.  kappa = max_m |(K_ZX W)_m|_1 is computed
   when a session is created (basq_recombine*, basq_features, basq_session_create); fp32 inputs with
   kappa > kappa_max (default 64, i.e. ~1e-5 of the outputscale; environment BASQ_F32_KAPPA_MAX; 0 = never)
   are promoted to the all-fp64 path inside the call - the reference's default likelihood noise 1e-10
   (BASQ/_parameters.py:30) makes such GPs easy to produce in low dimension.  kappa_max < 0 leaves the
   threshold unchanged; the outputs (may be NULL) report the last kappa and the number of promotions. */
int basq_ctx_conditioning(basq_ctx* ctx, double kappa_max, double* last_kappa_host, int64_t* promotions_host);
/* Opt-in for callers that hold fp64 arrays but accept fp32 kernel evaluation (SOBER runs in torch.double,
   SOBER/_settings.py:4-11): with on != 0, sessions created from fp64 inputs (basq_recombine*, basq_session_create)
   evaluate the kernel on the fp32 tensor-core path - narrowed copies of X, Z, Xobs; set sums, projection and
   Caratheodory stay fp64 exactly as for fp32 inputs - unless the conditioning guard above sends them back to
   fp64.  Kernel values then carry ~2e-7 relative error instead of 1e-16.  Default off (environment
   BASQ_F64_EVAL_F32=1).  on < 0 leaves the setting unchanged; demotions_host (may be NULL) receives the
   number of sessions demoted so far. */
int basq_ctx_allow_f32_eval(basq_ctx* ctx, int on, int64_t* demotions_host);
/* Key of the library's own Gaussian draws (the Nystrom test matrix when the caller passes none); the
   k-th draw after this call uses the Philox key seed + k.  Default 0. */
int basq_ctx_set_seed(basq_ctx* ctx, uint64_t seed);
/* number of kernels this library has launched on ctx so far (bench.py's gpu_launches) */
int64_t basq_ctx_launch_count(const basq_ctx* ctx);
/* kernel evaluations k(z, x) performed by the set-sum kernel on ctx so far (roofline accounting) */
int64_t basq_ctx_pair_evals(const basq_ctx* ctx);
/* CUDA-event timings (ms) accumulated per phase since the last reset:
   0 prepare, 1 set-sum, 2 projection GEMM, 3 Caratheodory, 4 apply/compact, 5 nystrom, 6 gp predict.
   Only recorded when enabled: event pairs are recorded on the stream without synchronising;
   basq_ctx_profile_read synchronises the stream and folds them in. */
int basq_ctx_profile(basq_ctx* ctx, int enable);
int basq_ctx_profile_read(basq_ctx* ctx, double* ms_host /*[8]*/, int64_t* calls_host /*[8]*/, int reset);

/* ---- kernel evaluations -------------------------------------------------------------------- */
/* out[a,b] (fp64) = kernel(X[a], Y[b]) in desc->mode.  Replaces the reference's kernel callable. */
int basq_gram(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t a,
              const void* Y, int64_t b, double* out);
/* GP posterior over candidates, predict() of BASQ/_gp.py:213-230 with exact variance.
   space 0: the warped GP itself (mean, var incl. likelihood noise);
   space 1: the model space of desc->mode (wsabil_predict / wsabim_predict / gspace_predict),
            `offset` is the WSABI alpha added to the mean.  var_out may be NULL. */
int basq_gp_predict(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N,
                    int space, double offset, double* mean_out, double* var_out);

/* ---- weighted double sums: SOBER's full_quadrature variance (SOBER/BASQ/_basq.py:48-81) ------ */
/* *out_host = a^T basq_gram(desc, X, X) a for weights a[N] (fp64, any sign, zeros allowed), without forming the
   N x N matrix: the kernel of desc->mode exactly as basq_gram evaluates it, including the diagonal terms
   (noise_diag, diag_add) of the square matrix.  The sum is accumulated in fp64 in a fixed order: the same
   inputs give the same bits on every call.  1 <= N < 2^31 - 1024; non-finite weights: BASQ_ERR_NUMERIC.
   Every mode.  fp32 inputs evaluate the kernel in fp32 (basq_ctx_allow_f32_eval applies to fp64 inputs as for
   sessions); in WSABI-M and MMLT the conditioning guard (basq_ctx_conditioning) computes kappa over every row
   of X and promotes fp32 inputs to the fp64 path beyond kappa_max.  The record buffer takes 64 B per point at
   d = 10 (fp32; 96 B fp64), so device memory limits N well below the index limit.  Synchronises. */
int basq_kernel_quadform(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N,
                         const double* a, double* out_host);
/* *out_host = sum_ij a_i b_j kernel(X[i], Y[j]) for X[N], Y[Mb] with weights a[N], b[Mb]: the kernel function
   alone.  X and Y are different arrays, so basq_gram's diagonal terms (noise_diag, diag_add) do not enter,
   even when Y is X.  Same conventions as basq_kernel_quadform. */
int basq_kernel_bilinear(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N, const double* a,
                         const void* Y, int64_t Mb, const double* b, double* out_host);

/* ---- Nystrom eigenbasis: ker_svd_sparsify, BASQ/_rchq.py:28-31 ------------------------------ */
/* Randomised range finder (Halko alg. 4.4, niter subspace iterations, as torch.svd_lowrank) on
   K(Z,Z) with the Gaussian test matrix Omega[M,q] (fp64): the caller's, or - Omega NULL, what
   torch.svd_lowrank does - drawn by the library on the device (basq_standard_normals with the key
   set by basq_ctx_set_seed plus the number of earlier draws).  U_out[q,M] has orthonormal rows
   spanning the captured range - an arbitrary orthonormal basis of it, NOT the singular vectors: no
   final rotation is applied, because recombination only depends on span(U) (the reference discards
   the singular values, BASQ/_rchq.py:36).  S_out[q] (may be NULL) receives the Rayleigh quotients
   u_i^T K u_i of the rows, unordered; do not truncate U by them. */
int basq_nystrom_basis(basq_ctx* ctx, const basq_kernel_desc* desc, const void* Z, int64_t M,
                       int q, const double* Omega, int niter, double* U_out, double* S_out);

/* ---- test functions ------------------------------------------------------------------------ */
/* Phi[N,q] (fp64) = (U @ kernel(Z, X))^T : the features whose moments recombination preserves. */
int basq_features(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N,
                  const void* Z, int64_t M, const double* U, int q, double* Phi_out);

/* ---- Caratheodory step: Tchernychova_Lyons_CAR, BASQ/_rchq.py:133-175 ------------------------ */
/* A[n, S] (ld = lda) holds UNNORMALISED barycentres: row 0 the set masses, rows 1.. the weighted
   feature sums.  Finds omega[S] >= 0 with at most n non-zeros and A omega = A 1 (i.e. the kept
   sets, each mass rescaled by omega_j).  A is destroyed.  n_kept_host may be NULL. */
int basq_car(basq_ctx* ctx, double* A, int n, int S, int lda, double* omega_out, int* n_kept_host);

/* Row-sharded variant for one process per GPU: rank `rank` of `world` evaluates, converts and multiplies only rows
   [rank * chunk, min(M, (rank + 1) * chunk)), chunk = ceil(M / world), of K(Z, Z); Z, Omega (or the seed, when
   Omega is NULL) must be the same on every rank.  The ranks meet through `exchange`, a function of the caller
   that the library calls on the host while its kernels are queued on the context's stream:
     op BASQ_XCHG_ALLREDUCE_GRAM: sum gram_buf[count] (fp64, count = q * q) over the ranks, in place;
     op BASQ_XCHG_ALLGATHER_ROWS: rows_buf is [world][count] (count = chunk * q); this rank's part is filled
                                  in, fetch the others'.
   Both must be ordered after the work already queued on the context's stream and before the work queued after
   they return (torch.distributed collectives on the current stream do this), and must return 0.  gram_buf
   [q * q] and rows_buf [world * chunk * q] are device buffers of the caller.  U_out [q, M] is the same basis
   on every rank.  The library itself links no communication library.  Same algorithm as basq_nystrom_basis;
   the Cholesky factorisations are replicated. */
#define BASQ_XCHG_ALLREDUCE_GRAM 0
#define BASQ_XCHG_ALLGATHER_ROWS 1
typedef int (*basq_exchange_fn)(void* user, int op, int64_t count);
int basq_nystrom_basis_sharded(basq_ctx* ctx, const basq_kernel_desc* desc, const void* Z, int64_t M, int q,
                               const double* Omega, int niter, int rank, int world, double* gram_buf,
                               double* rows_buf, basq_exchange_fn exchange, void* user, double* U_out);

/* ---- recombination: recombination / rc_kernel_svd / Mod_Tchernychova_Lyons, BASQ/_rchq.py:4-130 */
/* X[N,d] candidates, Z[M,d] landmarks, U[q,M] basis (fp64), mu[N] fp64 weights or NULL (uniform).
   Writes at most q+1 ascending indices and positive weights summing to sum(mu). */
int basq_recombine(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N,
                   const void* Z, int64_t M, const double* U, int q, const double* mu,
                   int64_t* idx_out, double* w_out, int* n_out_host);
/* Objective-aware recombination, SOBER/_rchq.py:67-69,138-146,177-196 (calc_obj): obj[N] (fp64) holds
   the reference's `obj = -calc_obj(samp)` per candidate.  Every Caratheodory level carries the
   objective as an extra row, keeps n + 1 columns, and then drops one more along the null direction of
   the moment rows that does not increase sum_i w_i obj_i: the rule preserves the same q + 1 moments
   with <= q + 1 points and an expected calc_obj at least that of the input measure. */
int basq_recombine_objective(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N,
                             const void* Z, int64_t M, const double* U, int q, const double* mu,
                             const double* obj, int64_t* idx_out, double* w_out, int* n_out_host);
/* One such level on A[n + 1, C] (ld = lda; row n = objective sums), omega_out[C]; A is destroyed. */
int basq_car_objective(basq_ctx* ctx, double* A, int n, int C, int lda, double* omega_out);
/* Same with HOST buffers for X, Z, U, mu and the outputs (the copies are part of the call);
   desc->Xobs / W / alpha stay device pointers (they belong to the GP model, not to the call).
   If U_host is NULL the basis is built on the device (basq_nystrom_basis) from Omega_host[M,q], or,
   when that is NULL too, from a test matrix drawn on the device - the reference's own call shape
   (recombination(pts_rec, pts_nys, ...) draws inside torch.svd_lowrank, BASQ/_rchq.py:28-31). */
int basq_recombine_host(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X_host, int64_t N,
                        const void* Z_host, int64_t M, const double* U_host, int q,
                        const double* Omega_host, int niter, const double* mu_host,
                        int64_t* idx_out_host, double* w_out_host, int* n_out_host);

/* ---- staged session: the same loop, one stage per call, for candidates sharded over ranks ---- */
/* Rank-local shard X[N_loc]; idx_base = global index of its first row; N_glob = total count
   (uniform weight 1/N_glob when mu == NULL).  Z, U and the GP caches are replicated. */
int basq_session_create(basq_ctx* ctx, const basq_kernel_desc* desc, const void* X, int64_t N_loc,
                        int64_t N_glob, int64_t idx_base, const void* Z, int64_t M,
                        const double* U, int q, const double* mu, basq_session** out);
/* The same from HOST candidates, for one process per GPU: basq_ctx_stage_candidates starts copying this rank's
   shard X_host[N_loc, d] (dtype) and, if not NULL, its weights mu_host[N_loc] from (pinned) host memory into a
   device buffer the context owns, on a side stream, and returns at once - call it first, build the basis
   (basq_nystrom_basis / _sharded) while the bytes travel, then basq_session_create_staged creates the
   session from the staged shard (it waits for the copy on the context's stream).  One staged shard per
   context at a time; basq_recombine_host uses the same buffer. */
int basq_ctx_stage_candidates(basq_ctx* ctx, const void* X_host, int64_t N_loc, int d, int dtype,
                              const double* mu_host);
int basq_session_create_staged(basq_ctx* ctx, const basq_kernel_desc* desc, int64_t N_loc, int64_t N_glob,
                               int64_t idx_base, const void* Z, int64_t M, const double* U, int q,
                               basq_session** out);
void basq_session_destroy(basq_session* s);
/* Objective-aware mode for a staged session: obj[N_loc] (device, fp64, -calc_obj per local row, kept
   by the caller) or NULL to switch it off.  Level systems then have n + 1 rows (basq_session_level
   writes [n + 1, S]) and are reduced with basq_car_objective.  Call before the first pass. */
int basq_session_set_objective(basq_session* s, const double* obj);
/* live local points (after dropping zero weights / after the last apply) */
int basq_session_count(const basq_session* s, int64_t* R_loc_host);
/* Local part of the round's barycentre system: A[n = q+1, S = 2n] (ld = S), columns >= min(S,R_glob)
   zero.  off_glob = number of live points on lower ranks.  Sum A over ranks before basq_car. */
int basq_session_partial(basq_session* s, int64_t R_glob, int64_t off_glob, double* A_out);
/* Rescale the kept sets by omega[S], drop the rest, compact.  Returns the new local count. */
int basq_session_apply(basq_session* s, int64_t R_glob, int64_t off_glob, const double* omega,
                       int64_t* R_loc_new_host);
/* surviving local points: global indices (ascending) and weights; cap = capacity of the outputs */
int basq_session_result(basq_session* s, int64_t* idx_out, double* w_out, int cap, int* n_out_host);

/* ---- refined passes: one sweep of kernel evaluations, log2(F) + 1 Caratheodory levels ------- */
/* A pass may refine every set j into the F cells j, j + S, ..., j + (F-1) S (cell of a point =
   global position mod F*S; F a power of two <= BASQ_MAX_CELL_FACTOR, R_glob >= F*S).  The cell sums
   G[:, c] = sum_{p in c} w_p k(Z, x_p) are linear in the points, so the set columns of the reference's
   round (BASQ/_rchq.py:81-101) are sums of cell columns, and after the round the two halves of every
   surviving set form the next round's sets WITHOUT new kernel evaluations: the candidates shrink by
   2F per sweep instead of 2.  Level l works on NODES: node u < S * 2^l = cells u + k * S * 2^l;
   its children at level l + 1 are u (low half) and u + S * 2^l (high half). */
/* F the library would pick for a pass over R_glob live points, R_loc_max = largest rank-local count */
int basq_session_cell_factor(const basq_session* s, int64_t R_glob, int64_t R_loc_max, int* F_out_host);
/* The sweep: cell sums and cell masses of this rank's live points (kept inside the session). */
int basq_session_pass_begin(basq_session* s, int64_t R_glob, int64_t off_glob, int F);
/* Local part of level lvl's system, A_out[n, S] (device, ld = S, unused columns zero): row 0 = masses,
   rows 1..q = U' G.  lvl 0: K columns, column i = set node_host[i] scaled by fpar_host[i] (ppos unused).
   lvl > 0: 2K columns [low halves | high halves] of the K survivors of level lvl - 1: node_host[i] =
   low child id, ppos_host[i] = the parent's column in level lvl - 1, fpar_host[i] = the parent's
   accumulated factor.  Levels must be requested in order.  Sum A over ranks, then basq_car. */
int basq_session_level(basq_session* s, int lvl, int K, const int* node_host, const int* ppos_host,
                       const double* fpar_host, double* A_out);
/* basq_session_level in two halves, for ranks that share the projection: fold writes the level's
   K set-sum columns of THIS rank's points, Gf_out[M_tot, K] (device, ld = ld_gf; M_tot = landmarks incl.
   appended observations, basq_session_landmarks); after a reduce-scatter of Gf by landmark rows over
   the ranks, project takes the summed rows [row0, row0 + nrows) (Gf_rows[nrows, K]) and writes this
   rank's part of the level system: U'[:, rows] Gf_rows plus its local masses.  The all-reduce of A
   that follows completes both sums; every rank has done 1/G of the projection flops. */
int basq_session_landmarks(const basq_session* s, int* Mtot_out_host);
int basq_session_level_fold(basq_session* s, int lvl, int K, const int* node_host, double* Gf_out, int64_t ld_gf);
int basq_session_level_project(basq_session* s, int lvl, int K, const int* node_host, const int* ppos_host,
                               const double* fpar_host, const double* Gf_rows, int64_t ld_gf, int row0,
                               int nrows, double* A_out);
/* Rescale the kept cells by factor_host[F*S] (HOST; product of the level factors along each cell's
   path, 0 = dropped), drop the rest, compact.  New local count out. */
int basq_session_apply_cells(basq_session* s, int64_t R_glob, int64_t off_glob, int F,
                             const double* factor_host, int64_t* R_loc_new_host);
/* ---- candidate side (SURVEY 8f): device sampling, prior density, importance weights --------- */
/* X_out[N, d] (dtype) = mean + L z, z ~ N(0, I): PriorSampler.__call__ (BASQ/_sampler.py:21-34,
   prior.sample) and SOBER Gaussian.sample (SOBER/_prior.py:107-118).  mean_host[d], chol_host[d, d]
   (lower Cholesky factor of the covariance, row-major) are HOST arrays.  Philox4x32-10, counter =
   (global row index, block of 4 dimensions), key = seed: row `offset + i` of the one stream defined
   by `seed` lands in X_out[i], so ranks sample disjoint shards by passing their first global row. */
int basq_sample_mvn(basq_ctx* ctx, uint64_t seed, int64_t offset, int64_t N, int d, int dtype,
                    const double* mean_host, const double* chol_host, void* X_out);
/* out[rows, cols] (fp64) ~ N(0, 1): the same stream with mean 0 and L = I, any number of columns (the
   test matrix R of torch.svd_lowrank, BASQ/_rchq.py:28-31). */
int basq_standard_normals(basq_ctx* ctx, uint64_t seed, int64_t offset, int64_t rows, int cols, double* out);
/* out[N] (fp64) = log N(x_i; mean, L L^T): prior.log_prob (BASQ/_sampler.py:136, 204-212),
   Gaussian.pdf (SOBER/_prior.py:120-131). */
int basq_mvn_logpdf(basq_ctx* ctx, const void* X, int64_t N, int d, int dtype, const double* mean_host,
                    const double* chol_host, double* out);
/* Weights over candidates from the GP moments mean[N], var[N] (basq_gp_predict), fp64 in and out.
   kind 0: UncertaintySampler.calc_weights (BASQ/_sampler.py:190-217): |m| / (ratio v + (1 - ratio) |m|)
           (or |m| / (ratio v) at ratio = 1) - the prior density cancels between f_rec and g_rec;
   kind 1: PI_BQ.lfi (SOBER/_pi.py:121-139): Phi((m - 1) / sqrt(v)), log(. + eps32) when log_out.
   normalise != 0 divides by the sum (uniform weights if the sum is zero or not finite). */
int basq_candidate_weights(basq_ctx* ctx, int kind, double ratio, int log_out, const double* mean,
                           const double* var, int64_t N, int normalise, double* w_out);
/* In place: w < eps -> 0, inf / nan -> eps, then normalise (uniform if the sum is 0):
   WeightsStabiliser.cleansing_weights (SOBER/_weights.py:21-38). */
int basq_cleanse_weights(basq_ctx* ctx, double* w, int64_t N, double eps);

/* Resampling without replacement proportional to w[N] (device, fp64, need not be normalised):
   UncertaintySampler.SIR = torch.multinomial(weights, n_return) (BASQ/_sampler.py:104-118), as an
   exponential race: key_i = -log(u_i) / w_i, u_i = Philox(seed; i); the n_out smallest keys in
   increasing order are n_out successive draws.  idx_out_host[n_out] (HOST) receives the indices in
   draw order, n_drawn_host their number (= min(n_out, #positive weights)). */
int basq_sir_resample(basq_ctx* ctx, const double* w, int64_t N, int64_t n_out, uint64_t seed,
                      int64_t* idx_out_host, int64_t* n_drawn_host);

/* ---- small dense helper exposed for tests ---------------------------------------------------- */
/* C[m,n] = alpha * op(A) op(B) + beta * C, fp64 row-major; op = transpose when the flag is set. */
int basq_dgemm(basq_ctx* ctx, int transA, int transB, int m, int n, int k, double alpha,
               const double* A, int lda, const double* B, int ldb, double beta, double* C, int ldc);

/* C[m,n] = A[m,k] B[n,k]^T on the tensor cores with fp32 accuracy (rows scaled by powers of two and split
   into fp16 hi + lo, three products, fp32 accumulation in TMEM: ~2^-21 relative to sum |a||b|).  fp64
   row-major in and out.  This is the GEMM behind the Nystrom subspace iteration and the posterior-covariance
   Gram correction for fp32 kernels. */
int basq_tgemm(basq_ctx* ctx, int m, int n, int k, const double* A, int lda, const double* B, int ldb,
               double* C, int ldc);

#ifdef __cplusplus
}
#endif
#endif /* BASQ_B200_H */
