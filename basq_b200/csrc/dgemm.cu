// fp64 GEMM for the per-round projection U' @ G (reference BASQ/_rchq.py:88), the GP cache products
// (K_ZX W, BASQ/_gp.py:270-273) and the Nystrom subspace iteration.
//
// There is no fp64 kind in tcgen05; on sm_100a the fp64 tensor path is the warp-level
// mma.sync.m8n8k4.f64 (DMMA), which runs at twice the DFMA-pipe rate measured on this part
// (a register-tiled DFMA version of this kernel topped out at 14 TFLOP/s).
// Accumulators in registers, operands through a three-stage cp.async pipeline (see below).  All four
// transpose combinations, arbitrary sizes and leading dimensions (16-byte copies when the operand
// is 16-byte aligned with an even leading dimension, 8-byte copies otherwise).
// Measured on B200 (999 x 11002 x 2000, the projection): 26.6 TFLOP/s; cuBLAS 12.9 reaches 33.2.
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"

namespace basq {

namespace {

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------------------------
// BK = 16, three cp.async stages (no register staging, one barrier per 16 k),
// warp grid WM x WN with MF x NF fragments per warp, so that the CTA tile (WM 8 MF) x (WN 8 NF) can
// be chosen per problem to fill the 148 SMs (128 x 112 gives 144 tiles for the 999 x 2000
// projection where 128 x 128 gives 128).  Shared layouts keep the operand's contiguous direction
// contiguous (16-byte copies) and pad the other stride to 4 (mod 16) doubles: every fragment load
// is conflict-free.
// ---------------------------------------------------------------------------------------------
#ifndef BASQ_DGEMM_PK
#define BASQ_DGEMM_PK 16
#endif
#ifndef BASQ_DGEMM_PST
#define BASQ_DGEMM_PST 3
#endif
constexpr int PK = BASQ_DGEMM_PK, PST = BASQ_DGEMM_PST;   // A/B: -DBASQ_DGEMM_PK=32

__device__ __forceinline__ void cp_async16(void* dst, const void* src, int bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async8(void* dst, const void* src, int bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src),
               "r"(bytes)
               : "memory");
}

// Stage one operand tile.  KCONT: the source is contiguous along k (tile stored [row][PK + 4]),
// otherwise along the row index (tile stored [k][R + 4]).  Out-of-range elements are zero-filled.
template <bool KCONT, int R, int NTHR>
__device__ __forceinline__ void stage_tile(double* sm, const double* __restrict__ P, int64_t ld, int r0, int Rmax, int k0,
                                           int K, int vec16, int tid) {
  constexpr int CHUNKS = R * PK / 2;
#pragma unroll
  for (int c0 = 0; c0 < CHUNKS; c0 += NTHR) {
    const int c = c0 + tid;
    if (CHUNKS % NTHR != 0 && c >= CHUNKS) break;
    int row, kk, inner_left;
    const double* src;
    double* dst;
    if (KCONT) {
      row = c / (PK / 2);
      kk = (c % (PK / 2)) * 2;
      const bool ok = r0 + row < Rmax;
      inner_left = ok ? K - (k0 + kk) : 0;
      src = P + (int64_t)(ok ? r0 + row : 0) * ld + k0 + kk;
      dst = sm + row * (PK + 4) + kk;
    } else {
      kk = c / (R / 2);
      row = (c % (R / 2)) * 2;
      const bool ok = k0 + kk < K;
      inner_left = ok ? Rmax - (r0 + row) : 0;
      src = P + (int64_t)(ok ? k0 + kk : 0) * ld + r0 + row;
      dst = sm + kk * (R + 4) + row;
    }
    const int n = inner_left >= 2 ? 2 : (inner_left == 1 ? 1 : 0);
    if (n == 0) src = P;
    if (vec16) {
      cp_async16(dst, src, n * 8);
    } else {
      cp_async8(dst, src, n >= 1 ? 8 : 0);
      cp_async8(dst + 1, n >= 2 ? src + 1 : P, n >= 2 ? 8 : 0);
    }
  }
}

template <bool TA, bool TB, int WM, int WN, int MF, int NF>
__global__ void __launch_bounds__(WM* WN * 32) dgemm_pipe_kernel(int M, int N, int K, double alpha,
                                                                const double* __restrict__ A, int64_t lda,
                                                                const double* __restrict__ B, int64_t ldb, double beta,
                                                                double* __restrict__ C, int64_t ldc, int tri_k, int a16,
                                                                int b16, int kchunk, double* __restrict__ part, int sym) {
  constexpr int BM = WM * 8 * MF, BNN = WN * 8 * NF, NTHR = WM * WN * 32;
  constexpr int AS = TA ? BM + 4 : PK + 4, BS = TB ? PK + 4 : BNN + 4;
  constexpr int A_EL = TA ? PK * (BM + 4) : BM * (PK + 4);
  constexpr int B_EL = TB ? BNN * (PK + 4) : PK * (BNN + 4);
  extern __shared__ __align__(16) double dg_smem[];
  double* As = dg_smem;
  double* Bs = dg_smem + PST * A_EL;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp / WN, wn = warp % WN;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BNN;
  if (sym && n0 >= m0 + BM) return;     // tile strictly above the diagonal: mirrored afterwards (sym 1) or left alone (2)
  if (tri_k & 1) K = min(K, n0 + BNN);  // op(B)[k][n] = 0 for k > n
  if (tri_k & 2) K = min(K, m0 + BM);   // op(A)[m][k] = 0 for k > m
  // split-K (small outputs, long K): slice blockIdx.z covers k in [kb, K) with K clipped to the slice
  const int kb = kchunk > 0 ? blockIdx.z * kchunk : 0;
  if (kchunk > 0) K = min(K, kb + kchunk);
  const int KT = K > kb ? (K - kb + PK - 1) / PK : 0;

  auto load = [&](int kt, int st) {
    stage_tile<!TA, BM, NTHR>(As + st * A_EL, A, lda, m0, M, kb + kt * PK, K, a16, tid);
    stage_tile<TB, BNN, NTHR>(Bs + st * B_EL, B, ldb, n0, N, kb + kt * PK, K, b16, tid);
  };

  double acc[MF][NF][2];
#pragma unroll
  for (int i = 0; i < MF; ++i)
#pragma unroll
    for (int j = 0; j < NF; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

#pragma unroll
  for (int s = 0; s < PST - 1; ++s) {
    if (s < KT) load(s, s);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  const int fr = lane >> 2, fk = lane & 3;
  for (int kt = 0; kt < KT; ++kt) {
    asm volatile("cp.async.wait_group %0;" ::"n"(PST - 2) : "memory");
    __syncthreads();
    if (kt + PST - 1 < KT) load(kt + PST - 1, (kt + PST - 1) % PST);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const double* as = As + (kt % PST) * A_EL;
    const double* bs = Bs + (kt % PST) * B_EL;
#pragma unroll
    for (int kc = 0; kc < PK / 4; ++kc) {
      double af[MF], bf[NF];
#pragma unroll
      for (int i = 0; i < MF; ++i) {
        const int r = wm * (8 * MF) + i * 8 + fr, k = kc * 4 + fk;
        af[i] = TA ? as[k * AS + r] : as[r * AS + k];
      }
#pragma unroll
      for (int j = 0; j < NF; ++j) {
        const int c = wn * (8 * NF) + j * 8 + fr, k = kc * 4 + fk;
        bf[j] = TB ? bs[c * BS + k] : bs[k * BS + c];
      }
#pragma unroll
      for (int i = 0; i < MF; ++i)
#pragma unroll
        for (int j = 0; j < NF; ++j) dmma(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
  }

#pragma unroll
  for (int i = 0; i < MF; ++i) {
    const int m = m0 + wm * (8 * MF) + i * 8 + fr;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < NF; ++j) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int n = n0 + wn * (8 * NF) + j * 8 + fk * 2 + h;
        if (n >= N) continue;
        if (part) {  // split-K: the raw partial sum of this slice; splitk_reduce_kernel finishes
          part[((int64_t)blockIdx.z * M + m) * N + n] = acc[i][j][h];
        } else {
          double* c = C + (int64_t)m * ldc + n;
          *c = (beta == 0.0) ? alpha * acc[i][j][h] : fma(alpha, acc[i][j][h], beta * (*c));
        }
      }
    }
  }
}

// C = alpha * (sum of the slices, in slice order: deterministic) + beta * C
// sym: entries above the diagonal take the sums of their mirror image (their own tiles were skipped)
__global__ void splitk_reduce_kernel(const double* __restrict__ part, int splits, int M, int N, double alpha,
                                     double beta, double* __restrict__ C, int64_t ldc, int sym) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)M * N) return;
  const int64_t r = t / N, cidx = t % N;
  const int64_t src = (sym && cidx > r) ? cidx * N + r : t;
  double s = 0.0;
  for (int z = 0; z < splits; ++z) s += part[(int64_t)z * M * N + src];
  double* c = C + (t / N) * ldc + (t % N);
  *c = (beta == 0.0) ? alpha * s : fma(alpha, s, beta * (*c));
}

// C[r][c] = C[c][r] for c > r (square, after a c_symmetric product without split-K)
__global__ void mirror_lower_kernel(double* __restrict__ C, int N, int64_t ldc) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)N * N) return;
  const int64_t r = t / N, c = t % N;
  if (c > r) C[r * ldc + c] = C[c * ldc + r];
}

template <bool TA, bool TB, int WM, int WN, int MF, int NF>
int launch_pipe(basq_ctx* ctx, int m, int n, int k, double alpha, const double* A, int64_t lda, const double* B,
                int64_t ldb, double beta, double* C, int64_t ldc, int tri_k, int sym, bool fixed_order = false) {
  constexpr int BM = WM * 8 * MF, BNN = WN * 8 * NF;
  constexpr int A_EL = TA ? PK * (BM + 4) : BM * (PK + 4);
  constexpr int B_EL = TB ? BNN * (PK + 4) : PK * (BNN + 4);
  constexpr int SMEM = PST * (A_EL + B_EL) * 8;
  auto kern = dgemm_pipe_kernel<TA, TB, WM, WN, MF, NF>;
  BASQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
  const int a16 = (lda % 2 == 0) && ((uintptr_t)A % 16 == 0), b16 = (ldb % 2 == 0) && ((uintptr_t)B % 16 == 0);
  dim3 grid((unsigned)ceil_div(n, BNN), (unsigned)ceil_div(m, BM));
  // split-K when the output has far fewer tiles than the GPU has SMs and K is long (e.g. the 99 x 200
  // projection of a batch of 100 over 10^4 landmarks, the q x q Gram matrices of CholeskyQR)
  int64_t tiles = (int64_t)grid.x * grid.y;
  if (sym) {  // only the tiles with n0 < m0 + BM do any work
    tiles = 0;
    for (unsigned by = 0; by < grid.y; ++by) tiles += std::min<int64_t>(grid.x, ceil_div64((int64_t)(by + 1) * BM, BNN));
  }
  int splits = 1;
  if (!fixed_order && sym != 2 && tri_k == 0 && tiles * 2 <= ctx->num_sms && k >= 16 * PK)
    splits = (int)std::min<int64_t>(ctx->num_sms / tiles, k / (8 * PK));
  if (splits <= 1) {
    kern<<<grid, WM * WN * 32, SMEM, ctx->stream>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, a16, b16, 0,
                                                    nullptr, sym);
    if (sym == 1) {
      mirror_lower_kernel<<<(unsigned)ceil_div64((int64_t)n * n, 256), 256, 0, ctx->stream>>>(C, n, ldc);
      ctx->launches++;
    }
    return BASQ_OK;
  }
  const int kchunk = ceil_div(ceil_div(k, splits), PK) * PK;
  splits = ceil_div(k, kchunk);
  DevBuf part;
  BASQ_TRY(part.alloc(ctx, sizeof(double) * (size_t)splits * m * n));
  grid.z = (unsigned)splits;
  kern<<<grid, WM * WN * 32, SMEM, ctx->stream>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, a16, b16, kchunk,
                                                  part.as<double>(), sym);
  splitk_reduce_kernel<<<(unsigned)ceil_div64((int64_t)m * n, 256), 256, 0, ctx->stream>>>(part.as<double>(), splits, m, n,
                                                                                          alpha, beta, C, ldc, sym);
  ctx->launches++;
  return BASQ_OK;  // `part` returns to the context's block cache; stream order keeps it intact until the reduction has run
}

// tile shape that needs the fewest SM-waves of work for an m x n output
template <bool TA, bool TB>
int launch_best(basq_ctx* ctx, int m, int n, int k, double alpha, const double* A, int64_t lda, const double* B,
                int64_t ldb, double beta, double* C, int64_t ldc, int tri_k, int sym, bool fixed_order) {
  // fixed_order: one tile shape and no split-K, so that every output element sums its k terms in the same order
  // whatever m and n are
  if (fixed_order)
    return launch_pipe<TA, TB, 2, 4, 8, 4>(ctx, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, sym, true);
  auto cost = [&](int bm, int bn) {
    const int64_t tiles = (int64_t)ceil_div(m, bm) * ceil_div(n, bn);
    return (double)ceil_div64(tiles, ctx->num_sms) * bm * bn;
  };
  // symmetric output: the smallest tile wastes the least work on the diagonal blocks and splits K most evenly
  if (sym) return launch_pipe<TA, TB, 2, 4, 4, 4>(ctx, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, sym);
  const double c0 = cost(128, 128), c1 = cost(128, 112), c2 = cost(64, 128);
  if (c1 < c0 && c1 <= c2) return launch_pipe<TA, TB, 4, 2, 4, 7>(ctx, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, 0);
  if (c2 < c0) return launch_pipe<TA, TB, 2, 4, 4, 4>(ctx, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, 0);
  return launch_pipe<TA, TB, 2, 4, 8, 4>(ctx, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, 0);
}

}  // namespace

int dgemm(basq_ctx* ctx, bool ta, bool tb, int m, int n, int k, double alpha, const double* A, int64_t lda,
          const double* B, int64_t ldb, double beta, double* C, int64_t ldc, bool b_lower_tri, bool a_lower_tri,
          bool c_symmetric, bool c_lower_only, bool fixed_order) {
  BASQ_CHECK(!c_symmetric || (m == n && beta == 0.0 && !b_lower_tri && !a_lower_tri), BASQ_ERR_INVALID,
             "dgemm: c_symmetric needs a square output, beta = 0 and dense operands");
  BASQ_CHECK(!c_lower_only || (m == n && !c_symmetric && !b_lower_tri && !a_lower_tri), BASQ_ERR_INVALID,
             "dgemm: c_lower_only needs a square output and dense operands");
  // A^T A and A A^T are recognised without the flag
  const bool gram = (ta != tb) && A == B && lda == ldb && m == n && beta == 0.0 && !b_lower_tri && !a_lower_tri;
  // sym 1: lower tiles, then mirrored; 2: lower tiles only
  const int sym = c_lower_only ? 2 : ((c_symmetric || gram) ? 1 : 0);
  const int tri_k = ((b_lower_tri && tb) ? 1 : 0) | ((a_lower_tri && !ta) ? 2 : 0);
  if (m <= 0 || n <= 0) return BASQ_OK;
  BASQ_CHECK(k >= 0, BASQ_ERR_INVALID, "dgemm: negative k");
  BASQ_CHECK(ceil_div(m, 64) <= 65535, BASQ_ERR_UNSUPPORTED, "dgemm: m=%d too large for one launch", m);
  if (!ta && !tb) BASQ_TRY((launch_best<false, false>(ctx, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, sym, fixed_order)));
  else if (ta && !tb) BASQ_TRY((launch_best<true, false>(ctx, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, sym, fixed_order)));
  else if (!ta && tb) BASQ_TRY((launch_best<false, true>(ctx, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, sym, fixed_order)));
  else BASQ_TRY((launch_best<true, true>(ctx, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, tri_k, sym, fixed_order)));
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

}  // namespace basq
