// Host-side dispatch of the set-sum kernel (see setsum_impl.cuh).
#include "setsum_impl.cuh"
#include "setsum_mma.cuh"

namespace basq {

int set_sums(basq_ctx* ctx, const KParams& kp, const SetSumArgs& a) {
  const RecPool& pool = *a.pool;
  const LmView& lm = a.lm;
  BASQ_CHECK(pool.dtype == lm.dtype && pool.dp == lm.dp, BASQ_ERR_INVALID, "set_sums: records/landmarks mismatch");
  BASQ_CHECK(a.p_lo >= 0 && a.p_hi <= pool.count && a.p_lo <= a.p_hi, BASQ_ERR_INVALID, "set_sums: bad point range");
  BASQ_CHECK(a.S >= 1, BASQ_ERR_INVALID, "set_sums: S must be positive");
  if (a.nl != NL_LIN) BASQ_CHECK(a.corrT != nullptr, BASQ_ERR_INVALID, "set_sums: non-linear mode needs corrT");
  ctx->pair_evals += (int64_t)lm.count * (a.p_hi - a.p_lo);
  SetSumDev dev;
  dev.recs = pool.buf[pool.cur].as<unsigned char>();
  dev.rec_bytes = pool.rec_bytes;
  dev.count = pool.count;
  dev.off = a.off_glob;
  dev.S = a.S;
  dev.p_lo = a.p_lo;
  dev.p_hi = a.p_hi;
  dev.zz = lm.zz;
  dev.bz = lm.b;
  dev.Mtot = lm.count;
  dev.os_f = kp.os_f;
  dev.os_d = kp.outputscale;
  dev.nl = a.nl;
  dev.corrT = a.corrT;
  dev.ld_corr = a.ld_corr;
  dev.sz = a.sz;
  dev.G = a.G;
  dev.ldg = a.ldg;
  dev.accumulate = a.accumulate ? 1 : 0;
  if (pool.dtype == BASQ_F32 && a.nl == NL_LIN && lm.lmA != nullptr) {
    // fp32 linear modes: argument tiles on the tensor cores (setsum_mma.cuh)
    SetSumMmaDev md;
    md.recs = dev.recs;
    md.count = dev.count;
    md.off = dev.off;
    md.S = dev.S;
    md.p_lo = dev.p_lo;
    md.p_hi = dev.p_hi;
    md.lmA = lm.lmA;
    md.Mtot = lm.count;
    md.n_mgroups = md.n_jgroups = 0;
    md.os_f = kp.os_f;
    md.G = dev.G;
    md.ldg = dev.ldg;
    md.accumulate = dev.accumulate;
    switch (kp.family) {
      case BASQ_RBF: return launch_setsum_mma_rbf(ctx, kp.dp, md);
      case BASQ_MATERN15: return launch_setsum_mma_m15(ctx, kp.dp, md);
      default: return launch_setsum_mma_m25(ctx, kp.dp, md);
    }
  }
  if (pool.dtype == BASQ_F32) {
    switch (kp.family) {
      case BASQ_RBF: return launch_setsum_f32_rbf(ctx, kp.dp, dev);
      case BASQ_MATERN15: return launch_setsum_f32_m15(ctx, kp.dp, dev);
      default: return launch_setsum_f32_m25(ctx, kp.dp, dev);
    }
  }
  switch (kp.family) {
    case BASQ_RBF: return launch_setsum_f64_rbf(ctx, kp.dp, dev);
    case BASQ_MATERN15: return launch_setsum_f64_m15(ctx, kp.dp, dev);
    default: return launch_setsum_f64_m25(ctx, kp.dp, dev);
  }
}

}  // namespace basq
