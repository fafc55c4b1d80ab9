// Weighted set sums of Gram columns - the dominant kernel of every Tchernychova-Lyons round
// (reference hot loop #1, BASQ/_rchq.py:81-86, restructured "sum first, project once").
//
//   G[m, j] (+)= sum over local points p with (off + p) mod S == j of  w_p * f( k(z_m, x_p) )
//
// Mapping (B200): a CTA of 128 threads owns 128*TM landmarks x JT consecutive sets; each thread
// keeps its TM landmarks in registers for the whole launch and TM*JT fp64 accumulators, and walks
// the set members e = 0,1,2,... (records p = j + e*S - off).  The JT records of one step are
// contiguous in HBM (JT * rec_bytes), staged into shared memory by a 3-stage cp.async ring and read
// back as warp-uniform (broadcast) 128-bit LDS, so global traffic is one pass over the records per
// landmark tile (L2-resident across tiles) and the SM is bound by FP32/MUFU issue, not by memory.
// fp32 kernel values are widened exactly and accumulated in fp64 (DFMA) - the moment-matching
// tolerance (1e-8) needs it.
#pragma once
#include "common.cuh"

namespace basq {

struct SetSumDev {
  const unsigned char* recs;
  int rec_bytes;
  int64_t count;  // local records
  int64_t off;    // global position of local record 0
  int S;
  int64_t p_lo, p_hi;
  const void* zz;  // f32: float [Mtot, DP] ; f64: double [Mtot, DP]
  const float* bz;
  int Mtot;
  float os_f;
  double os_d;
  int nl;
  const double* corrT;
  int64_t ld_corr;
  const double* sz;
  double* G;
  int64_t ldg;
  int accumulate;
  double grid_m;  // reproducible instances: 1.5 * 2^52 * Q of the pass's grid Q (grid_round, common.cuh)
  double grid_m2; // reproducible fp64 instances: the grid of the remainders term - hi, summed into G2
  double* G2;
};

__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gmem_src, bool valid) {
  const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(gmem_src), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

template <typename T, int DP>
struct SetSumCfg {
  // landmarks per thread: keep TM * DP * (regs per scalar) <= 96 registers
  static constexpr int W = sizeof(T) / 4;
  static constexpr int TM_RAW = 96 / (DP * W);
  static constexpr int TM = TM_RAW > 8 ? 8 : (TM_RAW < 1 ? 1 : TM_RAW);
  static constexpr int JT = 4;       // sets per CTA
  static constexpr int THREADS = 128;
  static constexpr int EC = 8;       // set members per pipeline stage
  static constexpr int NSTAGE = 3;
  static constexpr int RB = sizeof(T) == 4 ? ((24 + 4 * DP) + 15) / 16 * 16 : ((24 + 8 * DP) + 15) / 16 * 16;
  static constexpr int STAGE_BYTES = EC * JT * RB;
  static constexpr int SMEM_BYTES = NSTAGE * STAGE_BYTES;
};

// REPRO: every term is rounded to the pass's grid before it is added (see setsum_mma.cuh)
template <typename T, int FAM, int DP, bool NONLIN, bool REPRO>
__global__ void __launch_bounds__(128) setsum_kernel(const SetSumDev a) {
  using Cfg = SetSumCfg<T, DP>;
  constexpr int TM = Cfg::TM, JT = Cfg::JT, EC = Cfg::EC, NSTAGE = Cfg::NSTAGE, RB = Cfg::RB;
  extern __shared__ __align__(16) unsigned char smem[];

  const int tid = threadIdx.x;
  const int m0 = blockIdx.x * (Cfg::THREADS * TM);
  const int j0 = blockIdx.y * JT;

  // ---- landmarks of this thread -> registers
  T zreg[TM][DP];
  float breg[TM];
#pragma unroll
  for (int t = 0; t < TM; ++t) {
    const int m = m0 + t * Cfg::THREADS + tid;
    const bool ok = m < a.Mtot;
#pragma unroll
    for (int i = 0; i < DP; ++i) zreg[t][i] = ok ? reinterpret_cast<const T*>(a.zz)[(int64_t)m * DP + i] : (T)0;
    if constexpr (sizeof(T) == 4) breg[t] = ok ? a.bz[m] : 0.f; else breg[t] = 0.f;
  }
  double szreg[TM];
  if (NONLIN) {
#pragma unroll
    for (int t = 0; t < TM; ++t) {
      const int m = m0 + t * Cfg::THREADS + tid;
      szreg[t] = (m < a.Mtot && a.sz) ? a.sz[m] : 1.0;
    }
  }

  // fp64 inputs in reproducible instances: two grids, so that the fp64 accuracy of the terms survives - acc sums
  // the terms rounded to the grid of grid_m, acc2 their remainders rounded to the finer grid of grid_m2
  constexpr bool TWO = REPRO && sizeof(T) == 8;
  double acc[TM][JT];
  double acc2[TWO ? TM : 1][TWO ? JT : 1];
#pragma unroll
  for (int t = 0; t < TM; ++t)
#pragma unroll
    for (int jj = 0; jj < JT; ++jj) acc[t][jj] = 0.0;
#pragma unroll
  for (int t = 0; t < (TWO ? TM : 1); ++t)
#pragma unroll
    for (int jj = 0; jj < (TWO ? JT : 1); ++jj) acc2[t][jj] = 0.0;
  // term a * b on the two grids
  // (the remainder x y - hi is below Q / 2 and is rounded once by the fma)
  auto add2 = [&](int t, int jj, double x, double y) {
    const double hi = grid_round(x, y, a.grid_m);
    acc[t][jj] += hi;
    if constexpr (TWO) acc2[t][jj] += grid_round(__fma_rn(x, y, -hi), 1.0, a.grid_m2);
  };

  // ---- member range of this CTA: local p = j + e*S - off  in [p_lo, p_hi)
  const int64_t S = a.S;
  int64_t e_lo, e_hi;
  {
    const int64_t num_lo = a.p_lo + a.off - (int64_t)(j0 + JT - 1);
    e_lo = num_lo <= 0 ? 0 : (num_lo + S - 1) / S;
    const int64_t num_hi = a.p_hi - 1 + a.off - (int64_t)j0;
    e_hi = num_hi < 0 ? 0 : num_hi / S + 1;
  }
  const int64_t n_e = e_hi > e_lo ? e_hi - e_lo : 0;
  const int64_t n_chunks = (n_e + EC - 1) / EC;
  if (a.accumulate && n_e == 0) return;  // nothing of this point range falls into the CTA's sets (uniform over the CTA)

  auto load_chunk = [&](int64_t c, int stage) {
    if (c < n_chunks) {
      unsigned char* st = smem + stage * Cfg::STAGE_BYTES;
      constexpr int CH = EC * JT * (RB / 16);  // 16-byte pieces per stage
      for (int x = tid; x < CH; x += Cfg::THREADS) {
        const int piece = x % (RB / 16);
        const int slot = x / (RB / 16);  // ei * JT + jj
        const int jj = slot % JT;
        const int64_t e = e_lo + c * EC + slot / JT;
        const int64_t p = (int64_t)(j0 + jj) + e * S - a.off;
        const bool ok = (e < e_hi) && (j0 + jj < S) && (p >= a.p_lo) && (p < a.p_hi);
        const unsigned char* src = ok ? a.recs + p * RB + piece * 16 : a.recs;
        cp_async16_zfill(st + slot * RB + piece * 16, src, ok);
      }
    }
    cp_async_commit();
  };

#pragma unroll
  for (int s = 0; s < NSTAGE - 1; ++s) load_chunk(s, s);

  for (int64_t c = 0; c < n_chunks; ++c) {
    cp_async_wait<NSTAGE - 2>();
    __syncthreads();
    load_chunk(c + NSTAGE - 1, (int)((c + NSTAGE - 1) % NSTAGE));
    const unsigned char* st = smem + (int)(c % NSTAGE) * Cfg::STAGE_BYTES;
#pragma unroll 1
    for (int ei = 0; ei < EC; ++ei) {
#pragma unroll
      for (int jj = 0; jj < JT; ++jj) {
        const unsigned char* rec = st + (ei * JT + jj) * RB;
        const double2 hw = *reinterpret_cast<const double2*>(rec);  // wf, mu
        if constexpr (sizeof(T) == 4) {
          // floats from byte 16: [idx, a, x0 ...]
          constexpr int NF4 = (RB - 16) / 16;
          float f[NF4 * 4];
#pragma unroll
          for (int v = 0; v < NF4; ++v) {
            const float4 q = *reinterpret_cast<const float4*>(rec + 16 + v * 16);
            f[v * 4 + 0] = q.x; f[v * 4 + 1] = q.y; f[v * 4 + 2] = q.z; f[v * 4 + 3] = q.w;
          }
          const float pa = f[1];
          if (!NONLIN) {
#pragma unroll
            for (int t = 0; t < TM; ++t) {
              const float k = pair_eval_f32<FAM, DP>(&f[2], pa, reinterpret_cast<const float*>(zreg[t]), breg[t], a.os_f);
              if (REPRO) add2(t, jj, f2d_pos(k), hw.x);
              else acc[t][jj] = fma(f2d_pos(k), hw.x, acc[t][jj]);
            }
          } else {
            const int64_t e = e_lo + c * EC + ei;
            const int64_t p = (int64_t)(j0 + jj) + e * S - a.off;
            const bool ok = (e < e_hi) && (j0 + jj < S) && (p >= a.p_lo) && (p < a.p_hi);
            if (ok) {
              const double* crow = a.corrT + (p - a.p_lo) * a.ld_corr;
#pragma unroll
              for (int t = 0; t < TM; ++t) {
                const int m = m0 + t * Cfg::THREADS + tid;
                if (m < a.Mtot) {
                  const float k = pair_eval_f32<FAM, DP>(&f[2], pa, reinterpret_cast<const float*>(zreg[t]), breg[t], a.os_f);
                  const double cv = f2d_pos(k) - crow[m];
                  if (REPRO) add2(t, jj, nl_apply(a.nl, cv, szreg[t], hw.x), hw.y);
                  else acc[t][jj] = fma(nl_apply(a.nl, cv, szreg[t], hw.x), hw.y, acc[t][jj]);
                }
              }
            }
          }
        } else {
          // doubles from byte 16: [idx, x0, x1 ...]
          constexpr int ND2 = (RB - 16) / 16;
          double g[ND2 * 2];
#pragma unroll
          for (int v = 0; v < ND2; ++v) {
            const double2 q = *reinterpret_cast<const double2*>(rec + 16 + v * 16);
            g[v * 2 + 0] = q.x; g[v * 2 + 1] = q.y;
          }
          if (!NONLIN) {
#pragma unroll
            for (int t = 0; t < TM; ++t) {
              const double k = pair_eval_f64<FAM, DP>(&g[1], reinterpret_cast<const double*>(zreg[t]), a.os_d);
              if (REPRO) add2(t, jj, k, hw.x);
              else acc[t][jj] = fma(k, hw.x, acc[t][jj]);
            }
          } else {
            const int64_t e = e_lo + c * EC + ei;
            const int64_t p = (int64_t)(j0 + jj) + e * S - a.off;
            const bool ok = (e < e_hi) && (j0 + jj < S) && (p >= a.p_lo) && (p < a.p_hi);
            if (ok) {
              const double* crow = a.corrT + (p - a.p_lo) * a.ld_corr;
#pragma unroll
              for (int t = 0; t < TM; ++t) {
                const int m = m0 + t * Cfg::THREADS + tid;
                if (m < a.Mtot) {
                  const double k = pair_eval_f64<FAM, DP>(&g[1], reinterpret_cast<const double*>(zreg[t]), a.os_d);
                  const double cv = k - crow[m];
                  if (REPRO) add2(t, jj, nl_apply(a.nl, cv, szreg[t], hw.x), hw.y);
                  else acc[t][jj] = fma(nl_apply(a.nl, cv, szreg[t], hw.x), hw.y, acc[t][jj]);
                }
              }
            }
          }
        }
      }
    }
  }
  cp_async_wait<0>();

  // ---- write back
#pragma unroll
  for (int t = 0; t < TM; ++t) {
    const int m = m0 + t * Cfg::THREADS + tid;
    if (m >= a.Mtot) continue;
#pragma unroll
    for (int jj = 0; jj < JT; ++jj) {
      const int j = j0 + jj;
      if (j >= a.S) continue;
      double* dst = a.G + (int64_t)m * a.ldg + j;
      *dst = a.accumulate ? (*dst + acc[t][jj]) : acc[t][jj];
      if constexpr (TWO) {
        double* dst2 = a.G2 + (int64_t)m * a.ldg + j;
        *dst2 = a.accumulate ? (*dst2 + acc2[t][jj]) : acc2[t][jj];
      }
    }
  }
}

// host-side launcher for one (T, FAM): dispatch on the padded dimension
template <typename T, int FAM, int DP>
int launch_setsum_dp(basq_ctx* ctx, const SetSumDev& dev) {
  using Cfg = SetSumCfg<T, DP>;
  dim3 grid((unsigned)ceil_div(dev.Mtot, Cfg::THREADS * Cfg::TM), (unsigned)ceil_div(dev.S, Cfg::JT));
  BASQ_CHECK(grid.y <= 65535, BASQ_ERR_UNSUPPORTED, "set_sums: %d sets exceed the grid limit", dev.S);
  const bool repro = dev.grid_m != 0.0;
  if (dev.nl == NL_LIN && !repro)
    setsum_kernel<T, FAM, DP, false, false><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, ctx->stream>>>(dev);
  else if (!repro)
    setsum_kernel<T, FAM, DP, true, false><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, ctx->stream>>>(dev);
  else if (dev.nl == NL_LIN)
    setsum_kernel<T, FAM, DP, false, true><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, ctx->stream>>>(dev);
  else
    setsum_kernel<T, FAM, DP, true, true><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, ctx->stream>>>(dev);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

template <typename T, int FAM>
int launch_setsum_family(basq_ctx* ctx, int dp, const SetSumDev& dev) {
  switch (dp) {
    case 2: return launch_setsum_dp<T, FAM, 2>(ctx, dev);
    case 4: return launch_setsum_dp<T, FAM, 4>(ctx, dev);
    case 6: return launch_setsum_dp<T, FAM, 6>(ctx, dev);
    case 8: return launch_setsum_dp<T, FAM, 8>(ctx, dev);
    case 10: return launch_setsum_dp<T, FAM, 10>(ctx, dev);
    case 12: return launch_setsum_dp<T, FAM, 12>(ctx, dev);
    case 16: return launch_setsum_dp<T, FAM, 16>(ctx, dev);
    case 20: return launch_setsum_dp<T, FAM, 20>(ctx, dev);
    case 24: return launch_setsum_dp<T, FAM, 24>(ctx, dev);
    case 32: return launch_setsum_dp<T, FAM, 32>(ctx, dev);
  }
  set_error("set_sums: no kernel compiled for padded dimension %d", dp);
  return BASQ_ERR_UNSUPPORTED;
}

// one definition per translation unit (setsum_inst_*.cu)
int launch_setsum_f32_rbf(basq_ctx*, int, const SetSumDev&);
int launch_setsum_f32_m15(basq_ctx*, int, const SetSumDev&);
int launch_setsum_f32_m25(basq_ctx*, int, const SetSumDev&);
int launch_setsum_f64_rbf(basq_ctx*, int, const SetSumDev&);
int launch_setsum_f64_m15(basq_ctx*, int, const SetSumDev&);
int launch_setsum_f64_m25(basq_ctx*, int, const SetSumDev&);

}  // namespace basq
