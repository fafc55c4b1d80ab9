// Host side of the tensor-core set sums for the pairwise non-linear kernels (see nlsum.cuh):
// operand preparation (Az -> scaled fp16 hi / lo tiles), chunking of a pass over its set groups,
// dispatch of kxgen_kernel / nlsum_kernel.
#include <math.h>

#include <algorithm>

#include "nlsum2.cuh"

namespace basq {

namespace {

__global__ void d2f_kernel(const double* __restrict__ in, int n, float* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = (float)in[t];
}

}  // namespace

int launch_nlsum(basq_ctx* ctx, int fam, int nl, int dp, const NlsDev& dev, int mode) {
  const bool wm = (nl == NL_WSABIM);
  switch (fam) {
    case BASQ_RBF: return wm ? launch_nlsum_rbf_wm(ctx, dp, dev, mode) : launch_nlsum_rbf_ml(ctx, dp, dev, mode);
    case BASQ_MATERN15: return wm ? launch_nlsum_m15_wm(ctx, dp, dev, mode) : launch_nlsum_m15_ml(ctx, dp, dev, mode);
    default: return wm ? launch_nlsum_m25_wm(ctx, dp, dev, mode) : launch_nlsum_m25_ml(ctx, dp, dev, mode);
  }
}

int launch_nlsum2(basq_ctx* ctx, int fam, int nl, int dp, const NlsDev& dev) {
  const bool wm = (nl == NL_WSABIM);
  switch (fam) {
    case BASQ_RBF: return wm ? launch_nlsum2_rbf_wm(ctx, dp, dev) : launch_nlsum2_rbf_ml(ctx, dp, dev);
    case BASQ_MATERN15: return wm ? launch_nlsum2_m15_wm(ctx, dp, dev) : launch_nlsum2_m15_ml(ctx, dp, dev);
    default: return wm ? launch_nlsum2_m25_wm(ctx, dp, dev) : launch_nlsum2_m25_ml(ctx, dp, dev);
  }
}

int launch_kxgen(basq_ctx* ctx, int fam, int dp, const KxDev& dev) {
  switch (fam) {
    case BASQ_RBF: return launch_kxgen_rbf(ctx, dp, dev);
    case BASQ_MATERN15: return launch_kxgen_m15(ctx, dp, dev);
    default: return launch_kxgen_m25(ctx, dp, dev);
  }
}

int nls_prepare(basq_ctx* ctx, const KParams& kp, const double* Az, int M, int n_obs, const double* sz,
                NlOperands* op) {
  op->M = M;
  op->n_obs = n_obs;
  op->KP = ceil_div(n_obs, NLS_KB) * NLS_KB;
  op->n_mtiles = (ceil_div(M, 128) + 1) / 2 * 2;   // even: CTA pairs take two landmark tiles (nlsum2.cuh)
  op->kx_scale = ldexpf(1.f, NLS_KX_SHIFT - (int)ceil(log2(kp.outputscale)));
  const size_t halves = (size_t)op->n_mtiles * (op->KP / 8) * 128 * 8;
  BASQ_TRY(op->azh.alloc(ctx, halves * 2));
  BASQ_TRY(op->azl.alloc(ctx, halves * 2));
  BASQ_TRY(op->ainv.alloc(ctx, sizeof(float) * op->n_mtiles * 128));
  BASQ_TRY(op->szf.alloc(ctx, sizeof(float) * M));
  DevBuf rscale;
  BASQ_TRY(rscale.alloc(ctx, sizeof(float) * op->n_mtiles * 128));
  rowscale16_kernel<256><<<op->n_mtiles * 128, 256, 0, ctx->stream>>>(Az, M, n_obs, n_obs, op->kx_scale,
                                                                      rscale.as<float>(), op->ainv.as<float>());
  const int64_t tot = (int64_t)op->n_mtiles * (op->KP / 8) * 128;
  split16_kernel<128><<<(unsigned)ceil_div64(tot, 256), 256, 0, ctx->stream>>>(Az, M, n_obs, n_obs, op->KP, op->n_mtiles,
                                                                              rscale.as<float>(), op->azh.as<__half>(),
                                                                              op->azl.as<__half>());
  d2f_kernel<<<ceil_div(M, 256), 256, 0, ctx->stream>>>(sz, M, op->szf.as<float>());
  ctx->launches += 3;
  BASQ_CUDA(cudaGetLastError());
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));  // rscale goes out of scope
  return BASQ_OK;
}

// G[:, 0..S) = set sums of local records [p_lo, p_hi), set of a record = (off + p) mod S.
int nls_set_sums(basq_ctx* ctx, const KParams& kp, int nl, NlOperands* op, const RecPool& pool, const LmView& lmz,
                 const LmView& lmobs, int64_t off, int S, int64_t p_lo, int64_t p_hi, double* G, int64_t ldg) {
  BASQ_CHECK(pool.dtype == BASQ_F32 && lmz.dtype == BASQ_F32, BASQ_ERR_INVALID, "nlsum: fp32 records only");
  BASQ_CHECK(lmz.count == op->M && lmobs.count == op->n_obs, BASQ_ERR_INVALID, "nlsum: operand mismatch");
  BASQ_CHECK(p_lo >= 0 && p_hi <= pool.count && p_lo <= p_hi && S >= 1, BASQ_ERR_INVALID, "nlsum: bad range");
  if (p_hi == p_lo) {
    BASQ_CUDA(cudaMemsetAsync(G, 0, sizeof(double) * (size_t)op->M * ldg, ctx->stream));
    return BASQ_OK;
  }
  ctx->pair_evals += (int64_t)op->M * (p_hi - p_lo);
  // every cell has at most one member of the range: one column per cell (GRAM); else 8 sets x 32 members
  const bool gram = (p_hi - p_lo) <= (int64_t)S;
  const int JT = gram ? NLS_NT : NLS_JT, EC = NLS_NT / JT;
  // BASQ_NLS_2CTA=1: set sums on CTA pairs (tcgen05 cta_group::2, nlsum2.cuh).  Measured slower than the
  // one-CTA kernel (684 vs 625 ms for the config-5 sweep: tensor pipe 52 % vs 66 % active - the cross-CTA
  // full / empty hand-shake costs more than the halved B stream saves), so it stays opt-in.
  const bool pairs = !gram && ctx->num_sms >= 2 && ([] { const char* e = getenv("BASQ_NLS_2CTA"); return e && e[0] == '1'; }());
  const int n_jg_total = ceil_div(S, JT);
  // tile stride: an upper bound of any group's tile count.  The kernels start group g at
  // e_lo = ceil((p_lo + off - (g JT + JT - 1)) / S); the last group's column n_jg_total JT - 1 may exceed
  // S - 1 (GRAM mode with S < JT: 255), so the bound takes that column.
  const int64_t e_hi_max = (p_hi - 1 + off) / S + 1;
  const int64_t num_lo = p_lo + off - ((int64_t)n_jg_total * JT - 1);
  const int64_t e_lo_min = num_lo <= 0 ? 0 : (num_lo + S - 1) / S;
  const int T = (int)std::max<int64_t>(1, ceil_div64(e_hi_max - e_lo_min, EC));
  const size_t b_tile_bytes = (size_t)op->KP * NLS_NT * 2;              // one of hi / lo
  const size_t rec_tile_bytes = (size_t)NLS_NT * pool.rec_bytes;
  const size_t per_tile = 2 * b_tile_bytes + rec_tile_bytes;
  static const size_t budget = [] {
    const char* e = getenv("BASQ_NLS_CHUNK_MB");
    return (size_t)(e ? atoll(e) : 3072) << 20;
  }();
  int jg_chunk = (int)std::max<size_t>(1, budget / (per_tile * (size_t)T));
  jg_chunk = std::min(jg_chunk, n_jg_total);
  const size_t tiles_cap = (size_t)jg_chunk * T;
  if (op->cap_tiles < tiles_cap || op->cap_rec_bytes < rec_tile_bytes) {
    op->kxh.release(); op->kxl.release(); op->trec.release();
    BASQ_TRY(op->kxh.alloc(ctx, tiles_cap * b_tile_bytes));
    BASQ_TRY(op->kxl.alloc(ctx, tiles_cap * b_tile_bytes));
    BASQ_TRY(op->trec.alloc(ctx, tiles_cap * rec_tile_bytes));
    op->cap_tiles = tiles_cap;
    op->cap_rec_bytes = rec_tile_bytes;
  }
  // cells without a member in the range are not written by the kernels (GRAM mode writes valid slots only)
  BASQ_CUDA(cudaMemsetAsync(G, 0, sizeof(double) * (size_t)op->M * ldg, ctx->stream));
  for (int jg0 = 0; jg0 < n_jg_total; jg0 += jg_chunk) {
    const int n_jg = std::min(jg_chunk, n_jg_total - jg0);
    KxDev kx;
    kx.recs = pool.buf[pool.cur].as<unsigned char>();
    kx.off = off; kx.S = S; kx.p_lo = p_lo; kx.p_hi = p_hi;
    kx.jg0 = jg0; kx.n_jg = n_jg; kx.tiles_per_jg = T; kx.JT = JT; kx.EC = EC;
    kx.ozz = reinterpret_cast<const float*>(lmobs.zz); kx.obz = lmobs.b;
    kx.n_obs = op->n_obs; kx.KP = op->KP;
    kx.os_f = kp.os_f; kx.kx_scale = op->kx_scale;
    kx.split_half = pairs ? 1 : 0;
    kx.kxh = op->kxh.as<__half>(); kx.kxl = op->kxl.as<__half>(); kx.trec = op->trec.as<unsigned char>();
    BASQ_TRY(launch_kxgen(ctx, kp.family, kp.dp, kx));
    NlsDev d;
    d.off = off; d.S = S; d.p_lo = p_lo; d.p_hi = p_hi;
    d.jg0 = jg0; d.n_jg = n_jg; d.tiles_per_jg = T; d.JT = JT; d.EC = EC;
    d.azh = op->azh.as<__half>(); d.azl = op->azl.as<__half>(); d.ainv = op->ainv.as<float>();
    d.kxh = kx.kxh; d.kxl = kx.kxl; d.trec = kx.trec; d.KP = op->KP;
    d.zz = reinterpret_cast<const float*>(lmz.zz); d.bz = lmz.b; d.szf = op->szf.as<float>();
    d.M = op->M; d.n_mtiles = op->n_mtiles; d.os_f = kp.os_f;
    d.G = G; d.ldg = ldg;
    if (pairs) BASQ_TRY(launch_nlsum2(ctx, kp.family, nl, kp.dp, d));
    else BASQ_TRY(launch_nlsum(ctx, kp.family, nl, kp.dp, d, gram ? 1 : 0));
  }
  return BASQ_OK;
}

}  // namespace basq
