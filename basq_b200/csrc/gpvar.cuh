// Fused GP posterior variance over candidates on the tensor cores (fp32 inputs).
//
//   var(x) = sigma_f^2 + sigma_n^2 - k_x^T W k_x,   k_x = k(Xobs, x),  W = (K_XX + sigma_n^2 I)^-1
//   (predict() of BASQ/_gp.py:213-230 with the exact variance; consumers: calc_weights,
//    BASQ/_sampler.py:194-217; wsabim_predict, BASQ/_wsabi.py:265-277; gspace_predict,
//    SOBER/BASQ/_scale_mmlt.py:211-223; lfi, SOBER/_pi.py:121-139)
//
// "Batched triangular solves": with W = L^-T L^-1 (L the Cholesky factor of K_XX + sigma_n^2 I, recovered
// from W on the device, gpvar.cu) the quadratic form is |L^-1 k_x|^2, and v = L^-1 k_x over a tile of 128
// candidates is a GEMM against the explicit lower-triangular L^-1 whose result never leaves the SM:
//   D[p, o] = sum_{o' <= o} kx[p, o'] Linv[o, o']   tcgen05.mma kind::f16, M = 128 candidates (TMEM
//                                                   lanes), N = 256 observations, fp16 hi / lo split
//                                                   operands, three products (fp32 accuracy), the K
//                                                   loop stops at the diagonal block (half the flop);
//   epilogue: thread = candidate, sum_o D[p, o]^2 in fp32 blocks of 32, fp64 across blocks;
//             var = sigma_f^2 + sigma_n^2 - sum.
// Why L^-1 and not W: the rounding of a reduced-precision contraction scales with |M| |k|, and
// |k|^T |W| |k| reaches 1e4 on the benchmark GP (1002 observations in 10-D, cond 1.5e4) where
// 2 |v|^T |L^-1| |k| stays below 1e2: the T = tril(W + W^T) form measured 3e-3 absolute error, this one 1e-5.
//
// The kernel values k(Xobs, x) never leave the SM.  Eight generator warps (two threads per candidate of
// the tile) evaluate the kernel values of one 32-observation K block, split them into fp16 hi / lo and
// store them straight into the A stage in the tcgen05 K-major layout; the MMA warp contracts the stage
// against the L^-1 tiles of TWO observation column tiles at once (two 256-column accumulators = all of
// TMEM), so a K block is generated once per pair of column tiles (1.5x the unique evaluations at four
// column tiles; they cost a third of the MMA time and hide under it).  DRAM traffic: the candidates in
// (4 d B each), the variances out (8 B each).  The posterior mean rides along on the same kernel values.
//   warps 0-7   generators (measured: four warps generate as slowly as the MMAs run; eight hide under them)
//   warps 8-15  epilogue (TMEM lane quarter = warp % 4, two column halves)
//   warp 16     L^-1 tile producer (cp.async.bulk, 32 KB units: hi / lo of one column tile's K block)
//   warp 17     TMEM allocation + tcgen05.mma issue
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "nlsum.cuh"
#include "prep.cuh"

namespace basq {

constexpr int GPV_MT = 128;   // candidates per tile (MMA M)
constexpr int GPV_NT = 256;   // observations per column tile (MMA N)
constexpr int GPV_A_PIECE = (NLS_KB / 8) * GPV_MT * 16;   // 8 KB
constexpr int GPV_B_PIECE = (NLS_KB / 8) * GPV_NT * 16;   // 16 KB

constexpr int GPF_GEN_WARPS = 8, GPF_EPI_WARPS = 8;   // two generator threads per candidate row (16 of a K block's 32 observations each)
constexpr int GPF_THREADS = (GPF_GEN_WARPS + GPF_EPI_WARPS + 2) * 32;
constexpr int GPF_A_STAGE = 2 * GPV_A_PIECE;          // hi + lo of one generated K block: 16 KB
constexpr int GPF_B_STAGE = 2 * GPV_B_PIECE;          // hi + lo of ONE column tile's K block: 32 KB

struct GpfDev {
  const float* X;          // [n_points, d] raw candidates
  int64_t n_points;
  int n_ptiles;
  const float* ozz; const float* obz;     // prepared observations [n_obs, DP], [n_obs]
  int n_obs, KP;
  float kx_scale;
  const __half* th; const __half* tl;     // L^-1 tiles [KP / 256][KP / 8][256][8]
  const float* tinv;                      // [KP]
  double base;
  double* var_out;
  const double* alpha;                    // [n_obs] mean cache, or NULL
  double mean_c0;                         // mean constant
  double* mean_out;                       // [n_points] posterior mean c0 + sum_o alpha_o k(xobs_o, x), or NULL
};

template <int DP>
struct GpfCfg {
  // L^-1 pieces stream from L2 at the chip-wide cap (43 B/clk per SM): five 32 KB units in flight cover
  // ~3800 tensor-pipe cycles of latency (two 64 KB stages covered 1536 and left the pipe 47 % busy)
  static constexpr int NA = 2, NB = 5;
  static constexpr int OBF = (DP + 1 + 3) / 4 * 4;                   // floats per observation (zz[DP], b, padding): 128-bit loads
  static constexpr int OFF_A = 0;
  static constexpr int OFF_B = OFF_A + NA * GPF_A_STAGE;
  static constexpr int OFF_OBS = OFF_B + NB * GPF_B_STAGE;           // [2][32][OBF] floats
  static constexpr int OBS_BYTES = ((2 * NLS_KB * OBF * 4) + 15) / 16 * 16;
  static constexpr int OFF_ALPHA = OFF_OBS + OBS_BYTES;               // [2][32] doubles (mean cache of a K block)
  static constexpr int OFF_TINV = OFF_ALPHA + 2 * NLS_KB * 8;         // [8 epilogue warps][128] scale factors
  static constexpr int OFF_COMB = OFF_TINV + GPF_EPI_WARPS * (GPV_NT / 2) * 4;
  static constexpr int OFF_MEAN = OFF_COMB + 128 * 8;                 // [128] doubles: second generator thread's part
  static constexpr int OFF_BAR = OFF_MEAN + 128 * 8;
  static constexpr int SMEM_BYTES = OFF_BAR + 256;
  static_assert(SMEM_BYTES <= 227 * 1024, "gpvar (fused): shared memory budget");
};

template <int FAM, int DP>
__global__ void __launch_bounds__(GPF_THREADS, 1) gpvar_fused_kernel(KParams kp, const GpfDev a) {
  using Cfg = GpfCfg<DP>;
  constexpr int NA = Cfg::NA, NB = Cfg::NB, NT = GPV_NT, OBF = Cfg::OBF;
  extern __shared__ __align__(1024) unsigned char smem_gpf[];
  unsigned char* const smem = smem_gpf;
  float* sObs = reinterpret_cast<float*>(smem + Cfg::OFF_OBS);
  float* sTinv = reinterpret_cast<float*>(smem + Cfg::OFF_TINV);
  double* sAlpha = reinterpret_cast<double*>(smem + Cfg::OFF_ALPHA);
  double* sMean = reinterpret_cast<double*>(smem + Cfg::OFF_MEAN);
  double* sComb = reinterpret_cast<double*>(smem + Cfg::OFF_COMB);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* a_full = bars;                 // [NA] generator threads
  uint64_t* a_empty = a_full + NA;         // [NA] MMA commit
  uint64_t* b_full = a_empty + NA;         // [NB] tx
  uint64_t* b_empty = b_full + NB;         // [NB] MMA commit
  uint64_t* t_full = b_empty + NB;         // [2]
  uint64_t* t_empty = t_full + 2;          // [2] 8 epilogue warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < NA; ++s) {
      mma::mbar_init(&a_full[s], GPF_GEN_WARPS * 32);
      mma::mbar_init(&a_empty[s], 1);
    }
    for (int s = 0; s < NB; ++s) {
      mma::mbar_init(&b_full[s], 1);
      mma::mbar_init(&b_empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mma::mbar_init(&t_full[b], 1);
      mma::mbar_init(&t_empty[b], GPF_EPI_WARPS);
    }
    mma::fence_barrier_init();
  }
  if (warp == GPF_GEN_WARPS + GPF_EPI_WARPS + 1) mma::tmem_alloc(tmem_slot, 512);
  mma::tc_fence_before();
  __syncthreads();
  mma::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_ct = a.KP / NT;
  const int n_sweeps = (n_ct + 1) / 2;
  // K blocks up to the diagonal block of column tile c (L^-1 is lower triangular)
  auto nkb_of = [&](int c) { return min(a.KP, NT * (c + 1)) / NLS_KB; };

  if (warp < GPF_GEN_WARPS) {
    // ======================================================================== generators
    const int r = tid & (GPV_MT - 1), part = tid >> 7;   // candidate row of the tile, half of the K block
    constexpr int OBS_PER_THREAD = (NLS_KB * OBF + GPF_GEN_WARPS * 32 - 1) / (GPF_GEN_WARPS * 32);
    uint32_t it = 0, ob = 0;
    for (int i = tid; i < NLS_KB * OBF; i += GPF_GEN_WARPS * 32) {   // K block 0 -> buffer 0
      const int o = i / OBF, j = i % OBF;
      sObs[i] = (o < a.n_obs && j <= DP) ? (j < DP ? a.ozz[(size_t)o * DP + j] : a.obz[o]) : 0.f;
    }
    const bool want_mean = a.mean_out != nullptr;
    if (want_mean && tid < NLS_KB) sAlpha[tid] = tid < a.n_obs ? a.alpha[tid] : 0.0;
    mma::named_bar_sync(3, GPF_GEN_WARPS * 32);
    for (int item = blockIdx.x; item < a.n_ptiles; item += gridDim.x) {
      const int64_t p = (int64_t)item * GPV_MT + r;
      const bool ok = p < a.n_points;
      float x[DP];
      float pa = 0.f;
#pragma unroll
      for (int i = 0; i < DP; ++i) x[i] = 0.f;
      if (ok) {
        float xl[BASQ_MAX_DIM];
        float nrm;
        prep_point_f32(kp, a.X + p * kp.d, xl, &nrm);
#pragma unroll
        for (int i = 0; i < DP; ++i) x[i] = xl[i];
        pa = point_a_term(kp, nrm);
      }
      double msum = 0.0;   // posterior mean: accumulated in the last sweep, which visits every K block
      for (int sw = 0; sw < n_sweeps; ++sw) {
        const int c_last = min(2 * sw + 1, n_ct - 1);
        const int nkb = nkb_of(c_last);
        const bool acc_mean = want_mean && sw == n_sweeps - 1;
        for (int kb = 0; kb < nkb; ++kb, ++it, ++ob) {
          // The NEXT K block's observations are fetched into registers now and stored to the other
          // shared-memory buffer after this block's evaluations (an unprefetched fetch exposed ~800 cycles
          // of global-load latency per K block: long-scoreboard stalls, tensor pipe 47 % busy).  The
          // sequence of K blocks restarts at 0 with every sweep, so the block after the last one is block 0.
          const float* so = sObs + (ob & 1u) * (NLS_KB * OBF);
          float* so_next = sObs + ((ob + 1u) & 1u) * (NLS_KB * OBF);
          const int kb_next = (kb + 1 < nkb) ? kb + 1 : 0;
          float pre[OBS_PER_THREAD];
#pragma unroll
          for (int u = 0; u < OBS_PER_THREAD; ++u) {
            const int i = tid + u * (GPF_GEN_WARPS * 32);
            const int o = kb_next * NLS_KB + i / OBF, j = i % OBF;
            pre[u] = (i < NLS_KB * OBF && o < a.n_obs && j <= DP) ? (j < DP ? a.ozz[(size_t)o * DP + j] : a.obz[o]) : 0.f;
          }
          const double* sal = sAlpha + (ob & 1u) * NLS_KB;
          double pre_alpha = 0.0;
          if (want_mean && tid < NLS_KB && kb_next * NLS_KB + tid < a.n_obs) pre_alpha = a.alpha[kb_next * NLS_KB + tid];
          const int s = it % NA;
          mma::mbar_wait(&a_empty[s], ((it / NA) & 1u) ^ 1u);
          uint4* sh = reinterpret_cast<uint4*>(smem + Cfg::OFF_A + (size_t)s * GPF_A_STAGE) + r;
          uint4* sl = sh + GPV_A_PIECE / 16;
#pragma unroll
          for (int kq = 0; kq < NLS_KB / 16; ++kq) {
            const int kc = part * (NLS_KB / 16) + kq;
            __half2 h2[4], l2[4];
#pragma unroll
            for (int u = 0; u < 8; u += 2) {
              float vv[2];
#pragma unroll
              for (int w = 0; w < 2; ++w) {
                const int ol_ = kc * 8 + u + w;
                // the observation's coordinates arrive as broadcast 128-bit loads (scalar loads made the
                // generators LSU-bound: 11 wavefronts per evaluation next to the MMAs' own operand reads)
                float zo[OBF];
#pragma unroll
                for (int q4 = 0; q4 < OBF / 4; ++q4) {
                  const float4 w4 = *reinterpret_cast<const float4*>(&so[ol_ * OBF + q4 * 4]);
                  zo[q4 * 4 + 0] = w4.x; zo[q4 * 4 + 1] = w4.y; zo[q4 * 4 + 2] = w4.z; zo[q4 * 4 + 3] = w4.w;
                }
                float kv = pair_eval_f32<FAM, DP>(x, pa, zo, zo[DP], kp.os_f);
                kv = (ok && kb * NLS_KB + ol_ < a.n_obs) ? kv : 0.f;
                if (acc_mean) msum = fma(f2d_pos(kv), sal[ol_], msum);   // padded observations carry alpha = 0
                vv[w] = __fmul_rn(kv, a.kx_scale);
              }
              // hi = the value truncated to 11 significant bits (a mask, exactly representable in fp16), lo =
              // the exact fp32 remainder rounded to fp16; packed pair conversions only (scalar
              // float <-> half conversions share the 16-lane pipe of the ex2 and made it the bound)
              const float t0 = __uint_as_float(__float_as_uint(vv[0]) & 0xFFFFE000u);
              const float t1 = __uint_as_float(__float_as_uint(vv[1]) & 0xFFFFE000u);
              h2[u / 2] = __floats2half2_rn(t0, t1);
              l2[u / 2] = __floats2half2_rn(__fsub_rn(vv[0], t0), __fsub_rn(vv[1], t1));
            }
            sh[kc * GPV_MT] = *reinterpret_cast<const uint4*>(h2);
            sl[kc * GPV_MT] = *reinterpret_cast<const uint4*>(l2);
          }
          mma::fence_proxy_async();
          mma::mbar_arrive(&a_full[s]);
#pragma unroll
          for (int u = 0; u < OBS_PER_THREAD; ++u) {
            const int i = tid + u * (GPF_GEN_WARPS * 32);
            if (i < NLS_KB * OBF) so_next[i] = pre[u];
          }
          if (want_mean && tid < NLS_KB) sAlpha[((ob + 1u) & 1u) * NLS_KB + tid] = pre_alpha;
          mma::named_bar_sync(3, GPF_GEN_WARPS * 32);
        }
      }
      if (want_mean) {
        // the two generator threads of a row each summed half of every K block's observations
        if (part == 1) sMean[r] = msum;
        mma::named_bar_sync(3, GPF_GEN_WARPS * 32);
        if (part == 0 && ok) a.mean_out[p] = a.mean_c0 + (msum + sMean[r]);
        mma::named_bar_sync(3, GPF_GEN_WARPS * 32);
      }
    }
  } else if (warp < GPF_GEN_WARPS + GPF_EPI_WARPS) {
    // ======================================================================== epilogue
    const int ew = warp - GPF_GEN_WARPS;
    const int quarter = warp & 3, half = ew >> 2;   // TMEM lanes 32 (warp % 4) .. + 31
    const int row = quarter * 32 + lane;
    uint32_t use[2] = {0u, 0u};
    for (int item = blockIdx.x; item < a.n_ptiles; item += gridDim.x) {
      const int64_t p = (int64_t)item * GPV_MT + row;
      double acc = 0.0;
      for (int sw = 0; sw < n_sweeps; ++sw) {
        for (int i = 0; i < 2; ++i) {
          const int c = 2 * sw + i;
          if (c >= n_ct) break;
          // the 128 scale factors of this warp's column half, staged per column tile in the warp's own slot
          // (a table of all KP of them would bound the observation count); the __syncwarp before the
          // previous t_empty arrival ordered the previous tile's reads
          float* ti = sTinv + ew * (NT / 2);
          reinterpret_cast<float4*>(ti)[lane] = reinterpret_cast<const float4*>(a.tinv + c * NT + half * (NT / 2))[lane];
          __syncwarp();
          mma::mbar_wait(&t_full[i], use[i] & 1u);
          mma::tc_fence_after();
          const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + i * NT + half * (NT / 2);
#pragma unroll 1
          for (int cb = 0; cb < NT / 2; cb += 32) {
            uint32_t v[32];
            mma::tmem_ld32(taddr + cb, v);
            mma::tmem_ld_wait();
            float part = 0.f;
#pragma unroll
            for (int cc = 0; cc < 32; ++cc) {
              const float vo = __fmul_rn(__uint_as_float(v[cc]), ti[cb + cc]);
              part = __fmaf_rn(vo, vo, part);
            }
            acc += (double)part;
          }
          mma::tc_fence_before();
          __syncwarp();
          if (lane == 0) mma::mbar_arrive(&t_empty[i]);
          ++use[i];
        }
      }
      if (half == 1) sComb[row] = acc;
      mma::named_bar_sync(1, GPF_EPI_WARPS * 32);
      if (half == 0 && p < a.n_points) a.var_out[p] = a.base - (acc + sComb[row]);
      mma::named_bar_sync(2, GPF_EPI_WARPS * 32);
    }
  } else if (warp == GPF_GEN_WARPS + GPF_EPI_WARPS) {
    // ======================================================================== L^-1 tile producer
    if (lane == 0) {
      uint32_t it = 0;
      const size_t b_tile = (size_t)(a.KP / 8) * NT * 8;
      for (int item = blockIdx.x; item < a.n_ptiles; item += gridDim.x) {
        for (int sw = 0; sw < n_sweeps; ++sw) {
          const int c0 = 2 * sw, c1 = min(2 * sw + 1, n_ct - 1);
          const int nkb0 = nkb_of(c0), nkb = nkb_of(c1);
          for (int kb = 0; kb < nkb; ++kb) {
            const bool two = (c1 != c0);
            const size_t ko = (size_t)kb * (GPV_B_PIECE / 2);
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              if (i == 0 ? kb >= nkb0 : !two) continue;
              const int c = i == 0 ? c0 : c1;
              const int s = it % NB;
              mma::mbar_wait(&b_empty[s], ((it / NB) & 1u) ^ 1u);
              unsigned char* st = smem + Cfg::OFF_B + (size_t)s * GPF_B_STAGE;
              mma::mbar_expect_tx(&b_full[s], GPF_B_STAGE);
              mma::bulk_g2s(st, a.th + c * b_tile + ko, GPV_B_PIECE, &b_full[s]);
              mma::bulk_g2s(st + GPV_B_PIECE, a.tl + c * b_tile + ko, GPV_B_PIECE, &b_full[s]);
              ++it;
            }
          }
        }
      }
    }
  } else {
    // ======================================================================== MMA issuer
    constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(NT >> 3) << 17) | ((128u >> 4) << 24);
    uint32_t ita = 0, itb = 0, use[2] = {0u, 0u};
    for (int item = blockIdx.x; item < a.n_ptiles; item += gridDim.x) {
      for (int sw = 0; sw < n_sweeps; ++sw) {
        const int c0 = 2 * sw, c1 = min(2 * sw + 1, n_ct - 1);
        const bool two = (c1 != c0);
        const int nkb0 = nkb_of(c0), nkb = nkb_of(c1);
        mma::mbar_wait(&t_empty[0], (use[0] & 1u) ^ 1u);
        if (two) mma::mbar_wait(&t_empty[1], (use[1] & 1u) ^ 1u);
        mma::tc_fence_after();
        for (int kb = 0; kb < nkb; ++kb, ++ita) {
          const int sa = ita % NA;
          mma::mbar_wait(&a_full[sa], (ita / NA) & 1u);
          const uint32_t sta = mma::smem_u32(smem + Cfg::OFF_A + (size_t)sa * GPF_A_STAGE);
          const uint32_t ahi = sta, alo = sta + GPV_A_PIECE;
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            if (i == 0 ? kb >= nkb0 : !two) continue;
            const int sb = itb % NB;
            mma::mbar_wait(&b_full[sb], (itb / NB) & 1u);
            mma::tc_fence_after();
            if (lane == 0) {
              const uint32_t bhi = mma::smem_u32(smem + Cfg::OFF_B + (size_t)sb * GPF_B_STAGE), blo = bhi + GPV_B_PIECE;
              const uint32_t d = tmem_base + i * NT;
#pragma unroll
              for (int pr = 0; pr < 3; ++pr) {
                const uint32_t aa = (pr == 0) ? alo : ahi;
                const uint32_t bb = (pr == 1) ? blo : bhi;
#pragma unroll
                for (int ks = 0; ks < NLS_KB / 16; ++ks) {
                  const uint64_t ad = mma::smem_desc(aa + ks * 2 * (GPV_MT * 16), GPV_MT * 16, 128);
                  const uint64_t bd = mma::smem_desc(bb + ks * 2 * (NT * 16), NT * 16, 128);
                  umma_f16(d, ad, bd, IDESC, (kb > 0 || pr > 0 || ks > 0) ? 1u : 0u);
                }
              }
              mma::umma_commit(&b_empty[sb]);
            }
            __syncwarp();
            ++itb;
          }
          if (lane == 0) {
            mma::umma_commit(&a_empty[sa]);
            if (kb == nkb0 - 1) mma::umma_commit(&t_full[0]);
            if (two && kb == nkb - 1) mma::umma_commit(&t_full[1]);
          }
          __syncwarp();
        }
        ++use[0];
        if (two) ++use[1];
      }
    }
  }

  mma::tc_fence_before();
  __syncthreads();
  if (warp == GPF_GEN_WARPS + GPF_EPI_WARPS + 1) {
    mma::tc_fence_after();
    mma::tmem_dealloc(tmem_base, 512);
  }
}

template <int FAM, int DP>
int launch_gpvar_fused_dp(basq_ctx* ctx, const KParams& kp, const GpfDev& dev) {
  using Cfg = GpfCfg<DP>;
  BASQ_CHECK((size_t)Cfg::SMEM_BYTES <= ctx->smem_optin, BASQ_ERR_UNSUPPORTED,
             "gpvar: kernel needs %d B shared memory (limit %zu)", Cfg::SMEM_BYTES, ctx->smem_optin);
  if (dev.n_ptiles <= 0) return BASQ_OK;
  BASQ_CUDA(cudaFuncSetAttribute(gpvar_fused_kernel<FAM, DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  gpvar_fused_kernel<FAM, DP><<<std::min(ctx->num_sms, dev.n_ptiles), GPF_THREADS, Cfg::SMEM_BYTES, ctx->stream>>>(kp, dev);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

template <int FAM>
int launch_gpvar_fused_family(basq_ctx* ctx, const KParams& kp, const GpfDev& dev) {
  switch (kp.dp) {
    case 2: return launch_gpvar_fused_dp<FAM, 2>(ctx, kp, dev);
    case 4: return launch_gpvar_fused_dp<FAM, 4>(ctx, kp, dev);
    case 6: return launch_gpvar_fused_dp<FAM, 6>(ctx, kp, dev);
    case 8: return launch_gpvar_fused_dp<FAM, 8>(ctx, kp, dev);
    case 10: return launch_gpvar_fused_dp<FAM, 10>(ctx, kp, dev);
    case 12: return launch_gpvar_fused_dp<FAM, 12>(ctx, kp, dev);
    case 16: return launch_gpvar_fused_dp<FAM, 16>(ctx, kp, dev);
    case 20: return launch_gpvar_fused_dp<FAM, 20>(ctx, kp, dev);
    case 24: return launch_gpvar_fused_dp<FAM, 24>(ctx, kp, dev);
    case 32: return launch_gpvar_fused_dp<FAM, 32>(ctx, kp, dev);
  }
  set_error("gpvar: no kernel compiled for padded dimension %d", kp.dp);
  return BASQ_ERR_UNSUPPORTED;
}

int launch_gpvar_fused_rbf(basq_ctx*, const KParams&, const GpfDev&);
int launch_gpvar_fused_m15(basq_ctx*, const KParams&, const GpfDev&);
int launch_gpvar_fused_m25(basq_ctx*, const KParams&, const GpfDev&);

}  // namespace basq
