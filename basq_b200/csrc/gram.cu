// Kernel evaluations between prepared landmarks and raw points: base Gram blocks, landmark-weighted
// sums (GP posterior mean), posterior variance, and the per-point factors of the warped kernels.
// Reference: gpytorch ScaleKernel(RBF|Matern).forward as called from BASQ/_gp.py:213-277,
// BASQ/_wsabi.py:205-301, SOBER/BASQ/_scale_mmlt.py:211-278.
//
// These kernels take the dimension at run time (they are far from the round loop's cost); the fp32
// arithmetic repeats pair_eval_f32's operation sequence exactly, so values agree bit for bit with
// the set-sum kernel.
#include "common.cuh"
#include "prep.cuh"

namespace basq {

namespace {
constexpr int PT = 128;  // points per CTA (one per thread)
constexpr int LT = 32;   // landmarks staged per tile

// MODE 0: write out[m, p] ; MODE 1: accumulate coef[m] * k into a per-point fp64 sum
// FROMREC: the points are live candidate records (already centred and scaled), P = first record.
// DPM > 0 (fp32 only): the point's coordinates stay in registers (dp rounded up to DPM, a multiple of 4,
// padded with zeros: the extra fma(0, 0, acc) leave every bit of the result unchanged) and the staged
// landmarks are read back as broadcast 128-bit loads.
template <typename TIN, bool F64, int MODE, bool FROMREC, int DPM>
__global__ void __launch_bounds__(PT) landmark_point_kernel(KParams kp, const void* __restrict__ zz_,
                                                            const float* __restrict__ bz, int Mtot,
                                                            const TIN* __restrict__ P, int64_t npts,
                                                            double* __restrict__ out, int64_t ldo,
                                                            const double* __restrict__ coef, double c0,
                                                            int rec_bytes) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int dp = kp.dp;
  const int tid = threadIdx.x;
  const int64_t p = (int64_t)blockIdx.x * PT + tid;
  const bool pok = p < npts;

  if (!F64 && DPM > 0) {
    constexpr int D4 = DPM > 0 ? DPM : 4;
    float* zs = reinterpret_cast<float*>(smem_raw);          // [LT][D4]
    float* bs = zs + LT * D4;                                // [LT]
    float xr[D4];
#pragma unroll
    for (int i = 0; i < D4; ++i) xr[i] = 0.f;
    float nrm = 0.f, pa = 0.f;
    if (FROMREC) {
      if (pok) {
        const float* f = reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(P) + p * rec_bytes);
        pa = f[5];
#pragma unroll
        for (int i = 0; i < D4; ++i)
          if (i < dp) xr[i] = f[6 + i];
      }
    } else {
      if (pok) {
        float xl[BASQ_MAX_DIM];
        prep_point_f32(kp, P + p * kp.d, xl, &nrm);
#pragma unroll
        for (int i = 0; i < D4; ++i)
          if (i < dp) xr[i] = xl[i];
      }
      pa = point_a_term(kp, nrm);
    }
    const float* zz = reinterpret_cast<const float*>(zz_);
    double sum = 0.0;
    const int m_begin = (MODE == 0) ? blockIdx.y * LT : 0;
    const int m_end = (MODE == 0) ? min(Mtot, m_begin + LT) : Mtot;
    for (int mt = m_begin; mt < m_end; mt += LT) {
      __syncthreads();
      const int cnt = min(LT, m_end - mt);
      for (int x = tid; x < LT * D4; x += PT) {
        const int l = x / D4, i = x % D4;
        zs[x] = (l < cnt && i < dp) ? zz[(int64_t)(mt + l) * dp + i] : 0.f;
      }
      for (int x = tid; x < cnt; x += PT) bs[x] = bz[mt + x];
      __syncthreads();
      if (pok) {
        for (int l = 0; l < cnt; ++l) {
          float acc = __fadd_rn(pa, bs[l]);
          const float4* z4 = reinterpret_cast<const float4*>(zs + l * D4);
#pragma unroll
          for (int i4 = 0; i4 < D4 / 4; ++i4) {
            const float4 z = z4[i4];
            acc = __fmaf_rn(xr[4 * i4 + 0], z.x, acc);
            acc = __fmaf_rn(xr[4 * i4 + 1], z.y, acc);
            acc = __fmaf_rn(xr[4 * i4 + 2], z.z, acc);
            acc = __fmaf_rn(xr[4 * i4 + 3], z.w, acc);
          }
          const float k = finish_f32(kp.family, acc, kp.os_f);
          if (MODE == 0)
            out[(int64_t)(mt + l) * ldo + p] = f2d_pos(k);
          else
            sum = fma(f2d_pos(k), coef[mt + l], sum);
        }
      }
    }
    if (MODE == 1 && pok) out[p] = c0 + sum;
  } else if (!F64) {
    float* xs = reinterpret_cast<float*>(smem_raw);          // [dp][PT]
    float* zs = xs + dp * PT;                                // [LT][dp]
    float* bs = zs + LT * dp;                                // [LT]
    float xl[BASQ_MAX_DIM];
    float nrm = 0.f;
    float pa = 0.f;
    if (FROMREC) {
      if (pok) {
        const float* f = reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(P) + p * rec_bytes);
        pa = f[5];
        for (int i = 0; i < dp; ++i) xl[i] = f[6 + i];
      }
    } else {
      if (pok) prep_point_f32(kp, P + p * kp.d, xl, &nrm);
      pa = point_a_term(kp, nrm);
    }
    for (int i = 0; i < dp; ++i) xs[i * PT + tid] = pok ? xl[i] : 0.f;
    const float* zz = reinterpret_cast<const float*>(zz_);
    double sum = 0.0;
    const int m_begin = (MODE == 0) ? blockIdx.y * LT : 0;
    const int m_end = (MODE == 0) ? min(Mtot, m_begin + LT) : Mtot;
    for (int mt = m_begin; mt < m_end; mt += LT) {
      __syncthreads();
      const int cnt = min(LT, m_end - mt);
      for (int x = tid; x < cnt * dp; x += PT) zs[x] = zz[(int64_t)mt * dp + x];
      for (int x = tid; x < cnt; x += PT) bs[x] = bz[mt + x];
      __syncthreads();
      if (pok) {
        for (int l = 0; l < cnt; ++l) {
          float acc = __fadd_rn(pa, bs[l]);
          for (int i = 0; i < dp; ++i) acc = __fmaf_rn(xs[i * PT + tid], zs[l * dp + i], acc);
          const float k = finish_f32(kp.family, acc, kp.os_f);
          if (MODE == 0)
            out[(int64_t)(mt + l) * ldo + p] = f2d_pos(k);
          else
            sum = fma(f2d_pos(k), coef[mt + l], sum);
        }
      }
    }
    if (MODE == 1 && pok) out[p] = c0 + sum;
  } else {
    double* xs = reinterpret_cast<double*>(smem_raw);        // [dp][PT]
    double* zs = xs + dp * PT;                               // [LT][dp]
    double xl[BASQ_MAX_DIM];
    if (FROMREC) {
      if (pok) {
        const double* h = reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(P) + p * rec_bytes);
        for (int i = 0; i < dp; ++i) xl[i] = h[3 + i];
      }
    } else {
      if (pok) prep_point_f64(kp, P + p * kp.d, xl);
    }
    for (int i = 0; i < dp; ++i) xs[i * PT + tid] = pok ? xl[i] : 0.0;
    const double* zz = reinterpret_cast<const double*>(zz_);
    double sum = 0.0;
    const int m_begin = (MODE == 0) ? blockIdx.y * LT : 0;
    const int m_end = (MODE == 0) ? min(Mtot, m_begin + LT) : Mtot;
    for (int mt = m_begin; mt < m_end; mt += LT) {
      __syncthreads();
      const int cnt = min(LT, m_end - mt);
      for (int x = tid; x < cnt * dp; x += PT) zs[x] = zz[(int64_t)mt * dp + x];
      __syncthreads();
      if (pok) {
        for (int l = 0; l < cnt; ++l) {
          double r2 = 0.0;
          for (int i = 0; i < dp; ++i) {
            const double df = xs[i * PT + tid] - zs[l * dp + i];
            r2 = fma(df, df, r2);
          }
          const double k = finish_f64(kp.family, r2, kp.outputscale);
          if (MODE == 0)
            out[(int64_t)(mt + l) * ldo + p] = k;
          else
            sum = fma(k, coef[mt + l], sum);
        }
      }
    }
    if (MODE == 1 && pok) out[p] = c0 + sum;
  }
}

template <int MODE, bool FROMREC>
int launch_lp(basq_ctx* ctx, const KParams& kp, const LmView& lm, const void* P, int64_t npts, double* out,
              int64_t ldo, const double* coef, double c0, int rec_bytes) {
  if (npts <= 0 || lm.count <= 0) return BASQ_OK;
  const bool f64 = lm.dtype == BASQ_F64;
  const size_t esz = f64 ? 8 : 4;
  const size_t smem = esz * ((size_t)kp.dp * PT + (size_t)LT * kp.dp) + (f64 ? 0 : 4 * LT);
  const int64_t gx = ceil_div64(npts, PT);
  BASQ_CHECK(gx < (1ll << 31), BASQ_ERR_UNSUPPORTED, "too many points for one launch");
  dim3 grid((unsigned)gx, MODE == 0 ? (unsigned)ceil_div(lm.count, LT) : 1u);
  BASQ_CHECK(grid.y <= 65535, BASQ_ERR_UNSUPPORTED, "too many landmarks (%d) for one Gram launch", lm.count);
  if (f64) {
    landmark_point_kernel<double, true, MODE, FROMREC, 0><<<grid, PT, smem, ctx->stream>>>(
        kp, lm.zz, nullptr, lm.count, (const double*)P, npts, out, ldo, coef, c0, rec_bytes);
  } else {
    const int d4 = (kp.dp + 3) / 4 * 4;
#define BASQ_LP_CASE(D)                                                                                   \
  case D:                                                                                                \
    landmark_point_kernel<float, false, MODE, FROMREC, D><<<grid, PT, 4 * (LT * D + LT), ctx->stream>>>(  \
        kp, lm.zz, lm.b, lm.count, (const float*)P, npts, out, ldo, coef, c0, rec_bytes);                  \
    break;
    switch (d4) {
      BASQ_LP_CASE(4) BASQ_LP_CASE(8) BASQ_LP_CASE(12) BASQ_LP_CASE(16) BASQ_LP_CASE(20) BASQ_LP_CASE(24)
      BASQ_LP_CASE(28) BASQ_LP_CASE(32)
      default:
        landmark_point_kernel<float, false, MODE, FROMREC, 0><<<grid, PT, smem, ctx->stream>>>(
            kp, lm.zz, lm.b, lm.count, (const float*)P, npts, out, ldo, coef, c0, rec_bytes);
    }
#undef BASQ_LP_CASE
  }
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

// var[p] = base - sum_o V[o, p] * Y[o, p]
__global__ void coldot_kernel(const double* __restrict__ V, const double* __restrict__ Y, int rows, int64_t cols,
                              int64_t ld, double base, double* __restrict__ out) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= cols) return;
  double s = 0.0;
  for (int o = 0; o < rows; ++o) s = fma(V[(int64_t)o * ld + p], Y[(int64_t)o * ld + p], s);
  out[p] = base - s;
}

// T[i][k] = W[i][k] + W[k][i] (k < i), W[i][i] (k == i), 0 (k > i): v^T W v = sum_i v_i (T v)_i with a
// lower-triangular T - half the flops of W v for the posterior variance
__global__ void tri_fold_kernel(const double* __restrict__ W, int n, double* __restrict__ T) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)n * n) return;
  const int i = (int)(t / n), k = (int)(t % n);
  T[t] = k < i ? W[t] + W[(int64_t)k * n + i] : (k == i ? W[t] : 0.0);
}

// MMLT factor: mu_g = exp(m_h + v_h / 2) - 1   (SOBER/BASQ/_scale_mmlt.py:211-223)
__global__ void mmlt_factor_kernel(const double* __restrict__ mean, const double* __restrict__ var, int64_t n,
                                   double* __restrict__ out) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) out[p] = expm1(mean[p] + 0.5 * var[p]);
}
}  // namespace

int base_gram(basq_ctx* ctx, const KParams& kp, const LmView& lm, const void* P, int64_t b, double* out,
              int64_t ldo) {
  return launch_lp<0, false>(ctx, kp, lm, P, b, out, ldo, nullptr, 0.0, 0);
}

int base_gram_records(basq_ctx* ctx, const KParams& kp, const LmView& lm, const RecPool& pool, int64_t p_lo,
                      int64_t p_hi, double* out, int64_t ldo) {
  const unsigned char* first = pool.buf[pool.cur].as<unsigned char>() + p_lo * pool.rec_bytes;
  return launch_lp<0, true>(ctx, kp, lm, first, p_hi - p_lo, out, ldo, nullptr, 0.0, pool.rec_bytes);
}

int landmark_dot(basq_ctx* ctx, const KParams& kp, const LmView& lm, const double* coef, double c0, const void* P,
                 int64_t N, double* out) {
  return launch_lp<1, false>(ctx, kp, lm, P, N, out, 0, coef, c0, 0);
}

// mean[p] = c0 + sum_j G[p, j]  (the per-set partial sums of landmark_dot_tc)
__global__ void rowsum_cols_kernel(const double* __restrict__ G, int64_t n, int cols, double c0, double* __restrict__ out) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  double s = 0.0;
  for (int j = 0; j < cols; ++j) s += G[p * cols + j];
  out[p] = c0 + s;
}

int rowsum_cols(basq_ctx* ctx, const double* G, int64_t n, int cols, double c0, double* out) {
  rowsum_cols_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(G, n, cols, c0, out);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

// The same sum on the tensor-core set-sum kernel (setsum_mma.cuh) with the roles swapped: the N points are the
// "landmarks" (128 per tile row), the n_obs observations are the "records" carrying coef as their weight, spread
// over 8 sets so that the 256-column tiles are full; the 8 partial sums per point are added afterwards.
// 1e10 kernel evaluations (1e7 candidates x 1002 observations) take ~5 ms this way against ~12 ms on the
// CUDA-core kernel above - the per-candidate factors m(x) of the WSABI kernels (BASQ/_wsabi.py:216-224).
int landmark_dot_tc(basq_ctx* ctx, const KParams& kp, const void* Xobs, int n_obs, const double* coef, double c0,
                    const void* P, int64_t N, double* out) {
  constexpr int SETS = 8;
  constexpr int64_t CHUNK = 1 << 20;
  RecPool obs;
  BASQ_TRY(build_records(ctx, kp, BASQ_F32, Xobs, n_obs, 1.0, nullptr, coef, true, &obs));   // record weight = coef
  DevBuf G;
  BASQ_TRY(G.alloc(ctx, sizeof(double) * (size_t)std::min(CHUNK, N) * SETS));
  for (int64_t p0 = 0; p0 < N; p0 += CHUNK) {
    const int64_t cnt = std::min(CHUNK, N - p0);
    Landmarks lmx;
    BASQ_TRY(prep_landmarks(ctx, kp, BASQ_F32, static_cast<const float*>(P) + p0 * kp.d, cnt, nullptr, 0, &lmx));
    SetSumArgs a;
    a.pool = &obs;
    a.lm = lmx.view();
    a.off_glob = 0;
    a.S = SETS;
    a.p_lo = 0;
    a.p_hi = obs.count;
    a.nl = NL_LIN;
    a.corrT = nullptr;
    a.ld_corr = 0;
    a.sz = nullptr;
    a.G = G.as<double>();
    a.ldg = SETS;
    a.accumulate = false;
    BASQ_TRY(set_sums(ctx, kp, a));
    BASQ_TRY(rowsum_cols(ctx, G.as<double>(), cnt, SETS, c0, out + p0));
  }
  return BASQ_OK;
}

bool gpvar_route(basq_ctx* ctx, const basq_kernel_desc* desc) {
  { const char* t = getenv("BASQ_GPVAR"); ctx->no_gpvar = t && t[0] == '0'; }
  return desc->dtype == BASQ_F32 && !ctx->no_gpvar;
}

// Exact GP posterior mean / variance (likelihood noise included), BASQ/_gp.py:213-230.
int gp_predict_impl(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const LmView& lmobs,
                    const void* X, int64_t N, double* mean_out, double* var_out) {
  PhaseTimer timer(ctx, PH_GP);
  if (var_out && N > 0 && gpvar_route(ctx, desc)) {
    // fused tensor-core kernel: variance, and the mean from the same kernel values
    bool mean_done = false;
    BASQ_TRY(gp_variance_tc(ctx, desc, kp, lmobs, X, N, var_out, mean_out, &mean_done));
    if (mean_out && !mean_done) BASQ_TRY(landmark_dot(ctx, kp, lmobs, desc->alpha, desc->mean_const, X, N, mean_out));
    return BASQ_OK;
  }
  if (mean_out) {
    // the choice depends on the GP only, never on N: the per-point factors of the warped kernels must come out
    // bit-identical for the 1e7 candidates of a session and for the handful of points of a feature / Gram call
    if (desc->dtype == BASQ_F32 && N > 0 && desc->n_obs >= 64)
      BASQ_TRY(landmark_dot_tc(ctx, kp, desc->Xobs, desc->n_obs, desc->alpha, desc->mean_const, X, N, mean_out));
    else
      BASQ_TRY(landmark_dot(ctx, kp, lmobs, desc->alpha, desc->mean_const, X, N, mean_out));
  }
  if (!var_out || N == 0) return BASQ_OK;
  const int n_obs = desc->n_obs;
  // chunk so that V and Y (n_obs x P fp64 each) stay around 512 MB (large GEMMs: fewer, fuller waves)
  int64_t P = (int64_t)(512ll << 20) / (8ll * n_obs);
  P = P < 1024 ? 1024 : (P > 65536 ? 65536 : P);
  P = (P / 128) * 128;
  if (P > N) P = N;
  DevBuf V, Y, T;
  BASQ_TRY(V.alloc(ctx, sizeof(double) * n_obs * P));
  BASQ_TRY(Y.alloc(ctx, sizeof(double) * n_obs * P));
  BASQ_TRY(T.alloc(ctx, sizeof(double) * (size_t)n_obs * n_obs));
  tri_fold_kernel<<<(unsigned)ceil_div64((int64_t)n_obs * n_obs, 256), 256, 0, ctx->stream>>>(desc->W, n_obs, T.as<double>());
  ctx->launches++;
  const size_t esz = desc->dtype == BASQ_F64 ? 8 : 4;
  for (int64_t p0 = 0; p0 < N; p0 += P) {
    const int64_t cnt = (N - p0 < P) ? N - p0 : P;
    const void* Xc = (const unsigned char*)X + (size_t)p0 * desc->d * esz;
    BASQ_TRY(base_gram(ctx, kp, lmobs, Xc, cnt, V.as<double>(), P));
    BASQ_TRY(dgemm(ctx, false, false, n_obs, (int)cnt, n_obs, 1.0, T.as<double>(), n_obs, V.as<double>(), P, 0.0,
                   Y.as<double>(), P, /*b_lower_tri=*/false, /*a_lower_tri=*/true));
    coldot_kernel<<<ceil_div(cnt, 256), 256, 0, ctx->stream>>>(V.as<double>(), Y.as<double>(), n_obs, cnt, P,
                                                                desc->outputscale + desc->noise, var_out + p0);
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
  }
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));  // scratch goes out of scope
  return BASQ_OK;
}

// Per-point factor of the warped kernels: m(x) for WSABI-L/M, mu_g(x) for MMLT.
int warp_factor(basq_ctx* ctx, const basq_kernel_desc* desc, const KParams& kp, const LmView& lmobs,
                const void* X, int64_t N, double* out) {
  if (N == 0) return BASQ_OK;
  if (desc->mode == BASQ_WSABI_L || desc->mode == BASQ_WSABI_M)
    return gp_predict_impl(ctx, desc, kp, lmobs, X, N, out, nullptr);
  if (desc->mode == BASQ_MMLT_G) {
    DevBuf var;
    BASQ_TRY(var.alloc(ctx, sizeof(double) * N));
    BASQ_TRY(gp_predict_impl(ctx, desc, kp, lmobs, X, N, out, var.as<double>()));
    mmlt_factor_kernel<<<ceil_div(N, 256), 256, 0, ctx->stream>>>(out, var.as<double>(), N, out);
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
    // var is freed by cudaFree (synchronising) at scope exit, after the kernel was enqueued
    return BASQ_OK;
  }
  set_error("warp_factor: mode %d has no per-point factor", desc->mode);
  return BASQ_ERR_INVALID;
}

}  // namespace basq
