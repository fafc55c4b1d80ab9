// Host side of the fused posterior-variance kernel (gpvar.cuh): L^-1 recovered from W as row-scaled fp16
// hi / lo tiles, chunking over the candidates.
#include <math.h>

#include <algorithm>

#include "gpvar.cuh"

namespace basq {

// nystrom.cu
int spd_inverse_factor(basq_ctx* ctx, const double* A, int n, double* Linv_out);
int spd_chol_blocked(basq_ctx* ctx, double* A, int n);

namespace {
__global__ void zero_upper_kernel(double* __restrict__ A, int n) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)n * n) return;
  if ((int)(t % n) > (int)(t / n)) A[t] = 0.0;
}

// R[i, j] = W[n-1-i, n-1-j] for j <= i: the lower triangle of J W J, J the reversal permutation
__global__ void reverse_lower_kernel(const double* __restrict__ W, int n, double* __restrict__ R) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)n * n) return;
  const int i = (int)(t / n), j = (int)(t % n);
  if (j <= i) R[t] = W[(int64_t)(n - 1 - i) * n + (n - 1 - j)];
}

// Up to this padded size L^-1 is prepared as it always was (two inversions, below); the results of the
// variance path stay bit-identical there.  That is the only reason for two routes.
constexpr int GPV_TWO_INVERSION_KP = 4096;
}  // namespace

// var_out[N] = sigma_f^2 + sigma_n^2 - k_x^T W k_x for fp32 candidates X [N, d]
int gp_variance_tc(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const LmView& lmobs, const void* X,
                   int64_t N, double* var_out, double* mean_out, bool* mean_done) {
  if (mean_done) *mean_done = false;
  BASQ_CHECK(desc->dtype == BASQ_F32 && lmobs.dtype == BASQ_F32, BASQ_ERR_INVALID, "gpvar: fp32 inputs only");
  const int n_obs = desc->n_obs;
  BASQ_CHECK(n_obs <= GPV_MAX_OBS, BASQ_ERR_UNSUPPORTED,
             "gpvar: %d observations; the fp32 posterior variance takes at most %d", n_obs, GPV_MAX_OBS);
  const int KP = ceil_div(n_obs, GPV_NT) * GPV_NT;
  const int n_ct = KP / GPV_NT;
  const float kx_scale = ldexpf(1.f, NLS_KX_SHIFT - (int)ceil(log2(kp.outputscale)));
  // k^T W k = |L^-1 k|^2 with K = W^-1 = L L^T, W = L^-T L^-1
  const unsigned nn_grid = (unsigned)ceil_div64((int64_t)n_obs * n_obs, 256);
  const bool reversed = KP > GPV_TWO_INVERSION_KP;
  DevBuf Cinv, Kmat, Linv;
  BASQ_TRY(Linv.alloc(ctx, sizeof(double) * (size_t)n_obs * n_obs));
  if (!reversed) {
    // W = C C^T -> C^-1 ; K = W^-1 = C^-T C^-1 = L L^T -> L^-1
    BASQ_TRY(Cinv.alloc(ctx, sizeof(double) * (size_t)n_obs * n_obs));
    BASQ_TRY(Kmat.alloc(ctx, sizeof(double) * (size_t)n_obs * n_obs));
    BASQ_TRY(spd_inverse_factor(ctx, desc->W, n_obs, Cinv.as<double>()));
    zero_upper_kernel<<<nn_grid, 256, 0, ctx->stream>>>(Cinv.as<double>(), n_obs);
    ctx->launches++;
    BASQ_TRY(dgemm(ctx, true, false, n_obs, n_obs, n_obs, 1.0, Cinv.as<double>(), n_obs, Cinv.as<double>(), n_obs, 0.0,
                   Kmat.as<double>(), n_obs));
    BASQ_TRY(spd_inverse_factor(ctx, Kmat.as<double>(), n_obs, Linv.as<double>()));
    zero_upper_kernel<<<nn_grid, 256, 0, ctx->stream>>>(Linv.as<double>(), n_obs);
    ctx->launches++;
  } else {
    // One factorisation: W = L^-T L^-1 says that F = L^-1 (lower) is the factor of W = F^T F, i.e. the
    // Cholesky factor G of J W J (J the reversal permutation) reversed and transposed: L^-1 = J G^T J.
    // Linv holds G (lower triangle); rowscale16 / split16 read it through that index map.
    reverse_lower_kernel<<<nn_grid, 256, 0, ctx->stream>>>(desc->W, n_obs, Linv.as<double>());
    ctx->launches++;
    BASQ_TRY(spd_chol_blocked(ctx, Linv.as<double>(), n_obs));
  }
  DevBuf rscale, tinv, th, tl;
  BASQ_TRY(rscale.alloc(ctx, sizeof(float) * KP));
  BASQ_TRY(tinv.alloc(ctx, sizeof(float) * KP));
  const size_t t_halves = (size_t)n_ct * (KP / 8) * GPV_NT * 8;
  BASQ_TRY(th.alloc(ctx, t_halves * 2));
  BASQ_TRY(tl.alloc(ctx, t_halves * 2));
  const int64_t tot = (int64_t)n_ct * (KP / 8) * GPV_NT;
  if (!reversed) {
    rowscale16_kernel<256><<<KP, 256, 0, ctx->stream>>>(Linv.as<double>(), n_obs, n_obs, n_obs, kx_scale,
                                                        rscale.as<float>(), tinv.as<float>());
    split16_kernel<GPV_NT><<<(unsigned)ceil_div64(tot, 256), 256, 0, ctx->stream>>>(
        Linv.as<double>(), n_obs, n_obs, n_obs, KP, n_ct, rscale.as<float>(), th.as<__half>(), tl.as<__half>());
  } else {
    rowscale16_kernel<256, true><<<KP, 256, 0, ctx->stream>>>(Linv.as<double>(), n_obs, n_obs, n_obs, kx_scale,
                                                              rscale.as<float>(), tinv.as<float>());
    split16_kernel<GPV_NT, true><<<(unsigned)ceil_div64(tot, 256), 256, 0, ctx->stream>>>(
        Linv.as<double>(), n_obs, n_obs, n_obs, KP, n_ct, rscale.as<float>(), th.as<__half>(), tl.as<__half>());
  }
  ctx->launches += 2;
  BASQ_CUDA(cudaGetLastError());
  GpfDev f;
  f.X = reinterpret_cast<const float*>(X);
  f.n_points = N;
  f.n_ptiles = (int)ceil_div64(N, GPV_MT);
  f.ozz = reinterpret_cast<const float*>(lmobs.zz);
  f.obz = lmobs.b;
  f.n_obs = n_obs;
  f.KP = KP;
  f.kx_scale = kx_scale;
  f.th = th.as<__half>(); f.tl = tl.as<__half>();
  f.tinv = tinv.as<float>();
  f.base = desc->outputscale + desc->noise;
  f.var_out = var_out;
  f.alpha = desc->alpha;          // the posterior mean rides along: its kernel values are the same ones
  f.mean_c0 = desc->mean_const;
  f.mean_out = mean_out;
  if (mean_done) *mean_done = mean_out != nullptr;
  switch (kp.family) {
    case BASQ_RBF: BASQ_TRY(launch_gpvar_fused_rbf(ctx, kp, f)); break;
    case BASQ_MATERN15: BASQ_TRY(launch_gpvar_fused_m15(ctx, kp, f)); break;
    default: BASQ_TRY(launch_gpvar_fused_m25(ctx, kp, f)); break;
  }
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));  // scratch goes out of scope
  return BASQ_OK;
}

}  // namespace basq
