// Nystrom eigenbasis of the landmark Gram matrix (reference ker_svd_sparsify, BASQ/_rchq.py:28-31,
// i.e. torch.svd_lowrank(K, q, niter=2): Halko et al. 2009 alg. 4.4 range finder).
//
//   Y = K Omega ; Q = orth(Y) ; niter x { Q = orth(K^T Q) ; Q = orth(K Q) } ; U = Q^T
//
// Recombination only depends on span(U) (its test functions are U_i . k(Z, x); any invertible
// mixing of the rows leaves the set of feasible quadrature rules unchanged, and the Caratheodory
// kernel is invariant to row scaling), so the final small SVD of the reference - a rotation inside
// span(Q) - is replaced by Rayleigh quotients reported in S_out.
//
// orth() is shifted CholeskyQR3 in fp64: Gram matrix and triangular solve are GEMMs; the q x q
// Cholesky factor and its inverse come from one persistent cooperative kernel (row-distributed
// elimination of [G | I], one grid barrier per column).
#include <math.h>

#include <algorithm>
#include <utility>

#include "common.cuh"
#include "gridsync.cuh"
#include "tgemm.cuh"

namespace basq {

namespace {
constexpr int CH_THREADS = 512;

struct CholDev {
  double* G;     // [q, ld]  in: SPD matrix (upper part used) ; destroyed
  double* W;     // [q, ld]  out: L^-1 (lower triangular), G = L L^T
  int q;
  int64_t ld;
  double* prow;  // [2][2q]
  double floor;  // pivot floor
  unsigned* bar;
  int* status;
};

// Row k owned by CTA k % G.  Step k: owner scales row k of [G | W] by 1/sqrt(g_kk) and publishes it;
// every CTA eliminates column k from its rows below k.
__global__ void __launch_bounds__(CH_THREADS, 1) chol_inv_kernel(const CholDev a) {
  extern __shared__ __align__(16) double rowc[];  // [2q] cached pivot row
  __shared__ double bcast;
  __shared__ int abort_sh;
  const int q = a.q, G = gridDim.x, b = blockIdx.x, tid = threadIdx.x, NT = blockDim.x;
  unsigned target = 0;  // barriers passed

  // W = I on own rows
  for (int r = b; r < q; r += G)
    for (int c = tid; c < q; c += NT) a.W[(int64_t)r * a.ld + c] = (r == c) ? 1.0 : 0.0;
  __syncthreads();

  auto publish = [&](int k) {
    double* g = a.G + (int64_t)k * a.ld;
    double* w = a.W + (int64_t)k * a.ld;
    if (tid == 0) {
      double piv = g[k];
      if (!(piv > a.floor)) piv = a.floor;
      bcast = 1.0 / sqrt(piv);
    }
    __syncthreads();
    const double inv = bcast;
    double* pub = a.prow + (int64_t)(k & 1) * 2 * q;
    for (int c = tid; c < 2 * q; c += NT) {
      double v = 0.0;
      if (c < q) {
        if (c >= k) { v = g[c] * inv; g[c] = v; }
      } else {
        const int cw = c - q;
        if (cw <= k) { v = w[cw] * inv; w[cw] = v; }
      }
      __stcg(&pub[c], v);
    }
    __syncthreads();
  };
  auto update = [&](int r, int k) {
    double* g = a.G + (int64_t)r * a.ld;
    double* w = a.W + (int64_t)r * a.ld;
    if (tid == 0) bcast = g[k] / rowc[k];  // l_rk = g_rk / d_k  (rowc[k] = d_k)
    __syncthreads();
    const double l = bcast;
    if (l != 0.0) {
      for (int c = k + tid; c < q; c += NT) g[c] = (c == k) ? 0.0 : fma(-l, rowc[c], g[c]);
      for (int c = tid; c <= k; c += NT) w[c] = fma(-l, rowc[q + c], w[c]);
    }
    __syncthreads();
  };

  if (b == 0) publish(0);
  for (int k = 0; k < q; ++k) {
    if (grid_barrier(a.bar, target, a.status, &abort_sh)) return;
    const double* pub = a.prow + (int64_t)(k & 1) * 2 * q;
    for (int c = tid; c < 2 * q; c += NT) rowc[c] = __ldcg(&pub[c]);
    __syncthreads();
    const int kn = k + 1;
    if (kn < q && (kn % G) == b) {
      update(kn, k);
      publish(kn);
    }
    // own rows below k
    int r0 = kn + ((b - kn) % G + G) % G;
    for (int r = r0; r < q; r += G) {
      if (r == kn) continue;
      update(r, k);
    }
  }
}


// ---------------------------------------------------------------------------------------------
// Register-resident block version of the same elimination (the fast path for 2q <= 2048): CTA k
// keeps rows [kB, kB+B) of [G | I] in registers (thread t holds columns t, t+512, ...), performs its
// B diagonal pivots locally and streams the scaled rows to L2; one grid barrier per block; the CTAs
// below replay the B rank-1 updates.  See car2.cu for the same scheme with pivot search.
// ---------------------------------------------------------------------------------------------
constexpr int C2_NT = 512, C2_CPT = 4;

struct Chol2Dev {
  const double* G;  // [q, q]
  double* W;        // [q, q] out: L^-1
  int q;
  double* prow;     // [q][2q]
  double floor;
  unsigned* bar;
  int* status;
};

template <int B>
__global__ void __launch_bounds__(C2_NT, 1) chol2_kernel(const Chol2Dev a) {
  __shared__ double fbuf[2][8];
  __shared__ double pbcast[2];
  const int q = a.q, W2 = 2 * a.q, b = blockIdx.x, tid = threadIdx.x;
  int par = 0;
  const int r0 = b * B;
  const int rows_mine = max(0, min(B, q - r0));
  double reg[B][C2_CPT];
#pragma unroll
  for (int i = 0; i < B; ++i)
#pragma unroll
    for (int j = 0; j < C2_CPT; ++j) {
      const int c = tid + j * C2_NT;
      double v = 0.0;
      if (i < rows_mine && c < W2) v = (c < q) ? a.G[(int64_t)(r0 + i) * q + c] : ((c - q == r0 + i) ? 1.0 : 0.0);
      reg[i][j] = v;
    }

  // rows of the blocks above arrive through L2 ("the data is the flag", gridsync.cuh); a CTA is done
  // after its own block, so the loop ends at k == b
  for (int k = 0; k <= b; ++k) {
    const int kr0 = k * B;
    const int krows = min(B, q - kr0);
    if (b == k) {
#pragma unroll
      for (int i = 0; i < B; ++i) {
        if (i < krows) {
          const int r = kr0 + i;
          const int js = r / C2_NT;
          if ((r % C2_NT) == tid) {
            double p = 0.0;
#pragma unroll
            for (int j = 0; j < C2_CPT; ++j)
              if (j == js) p = reg[i][j];
            if (!(p > a.floor)) p = a.floor;
            const double inv = 1.0 / sqrt(p);
            pbcast[par] = inv;
            // multiplier of sibling row i2: g_i2r / d with d = p * inv the scaled diagonal
#pragma unroll
            for (int i2 = 0; i2 < B; ++i2) {
              double f = 0.0;
#pragma unroll
              for (int j = 0; j < C2_CPT; ++j)
                if (j == js) f = reg[i2][j];
              fbuf[par][i2] = f / (p * inv);
            }
          }
          __syncthreads();
          const double inv = pbcast[par];
#pragma unroll
          for (int j = 0; j < C2_CPT; ++j) {
            const int c = tid + j * C2_NT;
            reg[i][j] *= inv;
            if (c < W2) __stcg(&a.prow[(int64_t)r * W2 + c], reg[i][j]);
          }
#pragma unroll
          for (int i2 = 0; i2 < B; ++i2) {
            if (i2 > i && i2 < krows) {
              const double f = fbuf[par][i2];
#pragma unroll
              for (int j = 0; j < C2_CPT; ++j)
                reg[i2][j] = (tid + j * C2_NT == r) ? 0.0 : fma(-f, reg[i][j], reg[i2][j]);
            }
          }
          par ^= 1;
        }
      }
    } else {
      constexpr int PF = (B < 3) ? B : 3;
      double win[PF][C2_CPT];
#pragma unroll
      for (int i = 0; i < PF; ++i)
#pragma unroll
        for (int j = 0; j < C2_CPT; ++j) {
          const int c = tid + j * C2_NT;
          win[i][j] = (i < krows && c < W2) ? __ldcg(&a.prow[(int64_t)(kr0 + i) * W2 + c]) : 0.0;
        }
#pragma unroll
      for (int i = 0; i < B; ++i) {
        if (i < krows) {
          const int r = kr0 + i;
          // wait for row r; every missing word of rows r .. r+PF-1 is re-requested in ONE batch of
          // independent loads per L2 round trip (see car2.cu)
          for (int spins = 0;; ++spins) {
            bool ok = true;
#pragma unroll
            for (int j = 0; j < C2_CPT; ++j)
              if (tid + j * C2_NT < W2 && is_sentinel(win[i % PF][j])) ok = false;
            if (ok) break;
            if ((spins & 63) == 63 && (*reinterpret_cast<volatile int*>(a.status) != 0 || spins > BASQ_SPIN_LIMIT)) {
              if (spins > BASQ_SPIN_LIMIT) atomicExch(a.status, 2);
#pragma unroll
              for (int j = 0; j < C2_CPT; ++j) win[i % PF][j] = 0.0;
              break;
            }
#pragma unroll
            for (int w = 0; w < PF; ++w) {
              if (i + w < B && i + w < krows) {
#pragma unroll
                for (int j = 0; j < C2_CPT; ++j) {
                  const int c = tid + j * C2_NT;
                  if (c < W2 && is_sentinel(win[(i + w) % PF][j]))
                    win[(i + w) % PF][j] = __ldcg(&a.prow[(int64_t)(r + w) * W2 + c]);
                }
              }
            }
          }
          double cur[C2_CPT];
#pragma unroll
          for (int j = 0; j < C2_CPT; ++j) {
            const int c = tid + j * C2_NT;
            cur[j] = win[i % PF][j];
            if (i + PF < B) win[i % PF][j] = (i + PF < krows && c < W2) ? __ldcg(&a.prow[(int64_t)(r + PF) * W2 + c]) : 0.0;
          }
          const int js = r / C2_NT;
          if ((r % C2_NT) == tid) {
            double d = 1.0;
#pragma unroll
            for (int j = 0; j < C2_CPT; ++j)
              if (j == js) d = cur[j];
            const double invd = 1.0 / d;
#pragma unroll
            for (int i2 = 0; i2 < B; ++i2) {
              double f = 0.0;
#pragma unroll
              for (int j = 0; j < C2_CPT; ++j)
                if (j == js) f = reg[i2][j];
              fbuf[par][i2] = f * invd;
            }
          }
          __syncthreads();
#pragma unroll
          for (int i2 = 0; i2 < B; ++i2) {
            if (i2 < rows_mine) {
              const double f = fbuf[par][i2];
#pragma unroll
              for (int j = 0; j < C2_CPT; ++j)
                reg[i2][j] = (tid + j * C2_NT == r) ? 0.0 : fma(-f, cur[j], reg[i2][j]);
            }
          }
          par ^= 1;
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < B; ++i)
    if (i < rows_mine) {
#pragma unroll
      for (int j = 0; j < C2_CPT; ++j) {
        const int c = tid + j * C2_NT;
        if (c >= q && c < W2) a.W[(int64_t)(r0 + i) * q + (c - q)] = reg[i][j];
      }
    }
}

template <int B>
int launch_chol2(basq_ctx* ctx, const Chol2Dev& d, int grid) {
  void* args[] = {(void*)&d};
  BASQ_CUDA(cudaLaunchCooperativeKernel((const void*)chol2_kernel<B>, dim3(grid), dim3(C2_NT), args, 0, ctx->stream));
  return BASQ_OK;
}

__global__ void add_diag_kernel(double* __restrict__ G, int q, int64_t ld, double s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < q) G[(int64_t)i * ld + i] += s;
}

__global__ void diag_kernel(const double* __restrict__ T, int q, int64_t ld, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < q) out[i] = T[(int64_t)i * ld + i];
}

// out[0] = min_i |T_ii| / max_i |T_ii| of a triangular factor's diagonal (spread of the singular values behind it)
__global__ void diag_spread_kernel(const double* __restrict__ T, int q, int64_t ld, double* __restrict__ out) {
  __shared__ double lo[256], hi[256];
  double a = 1e300, b = 0.0;
  for (int i = threadIdx.x; i < q; i += 256) {
    const double v = fabs(T[(int64_t)i * ld + i]);
    a = fmin(a, v);
    b = fmax(b, v);
  }
  lo[threadIdx.x] = a;
  hi[threadIdx.x] = b;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) {
      lo[threadIdx.x] = fmin(lo[threadIdx.x], lo[threadIdx.x + w]);
      hi[threadIdx.x] = fmax(hi[threadIdx.x], hi[threadIdx.x + w]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = hi[0] > 0.0 ? lo[0] / hi[0] : 0.0;
}

// out[0] = trace(G)
__global__ void trace_kernel(const double* __restrict__ G, int q, int64_t ld, double* __restrict__ out) {
  __shared__ double sh[256];
  double s = 0.0;
  for (int i = threadIdx.x; i < q; i += 256) s += G[(int64_t)i * ld + i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = sh[0];
}

// out[1] = max |G - I| (how far the columns behind this Gram matrix are from orthonormal); one row per
// block, combined with an integer atomic max on the bit pattern (non-negative doubles order like
// unsigned integers, so the result does not depend on the order of arrival).  out[1] must be zeroed.
__global__ void gram_dev_kernel(const double* __restrict__ G, int q, int64_t ld, double* __restrict__ out) {
  __shared__ double sh[256];
  const int r = blockIdx.x;
  double dev = 0.0;
  for (int c = threadIdx.x; c < q; c += 256) dev = fmax(dev, fabs(G[(int64_t)r * ld + c] - (r == c ? 1.0 : 0.0)));
  sh[threadIdx.x] = dev;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + w]);
    __syncthreads();
  }
  if (threadIdx.x == 0)
    atomicMax(reinterpret_cast<unsigned long long*>(out + 1), (unsigned long long)__double_as_longlong(sh[0]));
}

// out [cols, rows] = in [rows, cols]^T (both row-major), 32 x 32 tiles through shared memory
__global__ void transpose_kernel(const double* __restrict__ in, int rows, int cols, double* __restrict__ out) {
  __shared__ double tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    if (r < rows && c < cols) tile[i][threadIdx.x] = in[(int64_t)r * cols + c];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (r < rows && c < cols) out[(int64_t)c * rows + r] = tile[threadIdx.x][i];
  }
}

struct OrthWs {
  DevBuf gram, linv, tmp, prow, prow2, flags, scal;
  // the Cholesky + inverse workspace of q x q factors; tmp [tmp_rows, q] and scal (orthonormalise's product
  // and scalars) only when tmp_rows > 0
  int alloc(basq_ctx* ctx, int q, int64_t tmp_rows) {
    BASQ_TRY(gram.alloc(ctx, sizeof(double) * (size_t)q * q));
    BASQ_TRY(linv.alloc(ctx, sizeof(double) * (size_t)q * q));
    BASQ_TRY(prow.alloc(ctx, sizeof(double) * 4 * q));
    BASQ_TRY(prow2.alloc(ctx, sizeof(double) * 2 * (size_t)q * q));
    BASQ_TRY(flags.alloc(ctx, 512));
    BASQ_CUDA(cudaMemsetAsync(flags.p, 0, 512, ctx->stream));   // the watchdog status (byte 256) stays set once fired
    if (tmp_rows > 0) {
      BASQ_TRY(tmp.alloc(ctx, sizeof(double) * (size_t)tmp_rows * q));
      BASQ_TRY(scal.alloc(ctx, 64));
    }
    return BASQ_OK;
  }
  // BASQ_ERR_NUMERIC if the grid barrier watchdog of a Cholesky kernel fired since alloc (synchronises)
  int check_status(basq_ctx* ctx, const char* who) {
    int status = 0;
    BASQ_CUDA(cudaMemcpyAsync(&status, flags.as<int>() + 64, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
    BASQ_CHECK(status == 0, BASQ_ERR_NUMERIC, "%s: grid barrier watchdog fired in the Cholesky kernel", who);
    return BASQ_OK;
  }
};

int chol_inverse(basq_ctx* ctx, OrthWs& ws, int q, double floor_val) {
  if (2 * q <= C2_NT * C2_CPT && q <= 8 * ctx->num_sms) {
    int B = 1;
    while (B < 8 && (q + B - 1) / B > ctx->num_sms) B *= 2;
    Chol2Dev d2;
    d2.G = ws.gram.as<double>();
    d2.W = ws.linv.as<double>();
    d2.q = q;
    d2.prow = ws.prow2.as<double>();
    d2.floor = floor_val;
    d2.bar = ws.flags.as<unsigned>();
    d2.status = ws.flags.as<int>() + 64;
    BASQ_CUDA(cudaMemsetAsync(ws.flags.p, 0, 256, ctx->stream));
    BASQ_CUDA(cudaMemsetAsync(ws.prow2.p, 0xFF, sizeof(double) * 2 * (size_t)q * q, ctx->stream));  // sentinel
    const int grid = (q + B - 1) / B;
    switch (B) {
      case 1: BASQ_TRY(launch_chol2<1>(ctx, d2, grid)); break;
      case 2: BASQ_TRY(launch_chol2<2>(ctx, d2, grid)); break;
      case 4: BASQ_TRY(launch_chol2<4>(ctx, d2, grid)); break;
      default: BASQ_TRY(launch_chol2<8>(ctx, d2, grid)); break;
    }
    ctx->launches++;
    return BASQ_OK;
  }
  CholDev d;
  d.G = ws.gram.as<double>();
  d.W = ws.linv.as<double>();
  d.q = q;
  d.ld = q;
  d.prow = ws.prow.as<double>();
  d.floor = floor_val;
  d.bar = ws.flags.as<unsigned>();
  d.status = ws.flags.as<int>() + 64;
  BASQ_CUDA(cudaMemsetAsync(ws.flags.p, 0, 256, ctx->stream));
  const size_t smem = sizeof(double) * 2 * q;
  BASQ_CHECK(smem <= ctx->smem_optin, BASQ_ERR_UNSUPPORTED, "nystrom: q=%d too large for the Cholesky kernel", q);
  BASQ_CUDA(cudaFuncSetAttribute(chol_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int G = (q + 1) / 2;
  if (G > ctx->num_sms) G = ctx->num_sms;
  if (G < 1) G = 1;
  void* args[] = {(void*)&d};
  BASQ_CUDA(cudaLaunchCooperativeKernel((const void*)chol_inv_kernel, dim3(G), dim3(CH_THREADS), args, smem,
                                        ctx->stream));
  ctx->launches++;
  return BASQ_OK;
}

// Y [M, q] (ld = q) <- basis of span(Y) by shifted CholeskyQR: `passes` = 3 gives an orthonormal
// basis to machine precision (sCholQR3); 2 is enough between subspace iterations, where only the
// conditioning of the basis matters.  M_glob = rows of the whole matrix (the shift depends on it).
// `sh` (row-sharded basis): Y holds this rank's M rows only; the Gram matrix is summed over the ranks through the
// caller's exchange function, everything after it (trace, shift, Cholesky + inverse) is replicated and the
// factor is applied to the local rows.
int orthonormalise(basq_ctx* ctx, OrthWs& ws, double* Y, int64_t M, int q, int passes, int64_t M_glob,
                   const NysShard* sh) {
  // passes < 0: "until orthonormal to fp64" - a pass whose input Gram matrix is within 0.1 of the
  // identity is the last one (CholeskyQR squares the distance to orthonormality); at most 4.
  const bool adaptive = passes < 0;
  if (adaptive) passes = 4;
  for (int pass = 0; pass < passes; ++pass) {
    if (M > 0) {
      BASQ_TRY(dgemm(ctx, true, false, q, q, (int)M, 1.0, Y, q, Y, q, 0.0, ws.gram.as<double>(), q, false, false,
                     /*c_symmetric=*/true));
    } else {
      BASQ_CUDA(cudaMemsetAsync(ws.gram.p, 0, sizeof(double) * (size_t)q * q, ctx->stream));
    }
    if (sh) {   // sum of the ranks' partial Gram matrices (identical bits on every rank afterwards)
      BASQ_CUDA(cudaMemcpyAsync(sh->gram_buf, ws.gram.p, sizeof(double) * (size_t)q * q, cudaMemcpyDeviceToDevice, ctx->stream));
      BASQ_CHECK(sh->fn(sh->user, BASQ_XCHG_ALLREDUCE_GRAM, (int64_t)q * q) == 0, BASQ_ERR_INVALID,
                 "nystrom: the exchange function failed (all-reduce of the Gram matrix)");
      BASQ_CUDA(cudaMemcpyAsync(ws.gram.p, sh->gram_buf, sizeof(double) * (size_t)q * q, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    BASQ_CUDA(cudaMemsetAsync(ws.scal.p, 0, 2 * sizeof(double), ctx->stream));
    trace_kernel<<<1, 256, 0, ctx->stream>>>(ws.gram.as<double>(), q, q, ws.scal.as<double>());
    ctx->launches++;
    if (adaptive && pass > 0) {
      gram_dev_kernel<<<q, 256, 0, ctx->stream>>>(ws.gram.as<double>(), q, q, ws.scal.as<double>());
      ctx->launches++;
    }
    double trdev[2] = {0.0, 0.0};
    BASQ_CUDA(cudaMemcpyAsync(trdev, ws.scal.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
    const double tr = trdev[0];
    BASQ_CHECK(isfinite(tr) && tr > 0.0, BASQ_ERR_NUMERIC, "nystrom: Gram trace %g is not positive/finite", tr);
    if (adaptive && pass > 0 && trdev[1] < 0.1) passes = pass + 1;  // this pass finishes the job
    const double eps = 2.220446049250313e-16;
    // shift of Fukaya et al. (shifted CholeskyQR3): 11 (M q + q (q+1)) u |Y|_2^2 ; |Y|_2^2 <= trace
    const double shift = (pass == 0) ? 11.0 * ((double)M_glob * q + (double)q * (q + 1)) * eps * tr : 0.0;
    if (shift > 0.0) {
      add_diag_kernel<<<ceil_div(q, 256), 256, 0, ctx->stream>>>(ws.gram.as<double>(), q, q, shift);
      ctx->launches++;
    }
    BASQ_TRY(chol_inverse(ctx, ws, q, tr * 1e-30));
    // Y <- Y L^-T
    if (M > 0) {
      BASQ_TRY(dgemm(ctx, false, true, (int)M, q, q, 1.0, Y, q, ws.linv.as<double>(), q, 0.0, ws.tmp.as<double>(), q,
                     /*b_lower_tri=*/true));
      BASQ_CUDA(cudaMemcpyAsync(Y, ws.tmp.p, sizeof(double) * (size_t)M * q, cudaMemcpyDeviceToDevice, ctx->stream));
    }
  }
  return ws.check_status(ctx, "nystrom");
}

}  // namespace

// Linv_out [n, n] (row-major, fp64) = L^-1 with A = L L^T for a symmetric positive definite A [n, n]:
// the cooperative Cholesky + inverse kernels of the CholeskyQR step, on their own (gpvar.cu).
int spd_inverse_factor(basq_ctx* ctx, const double* A, int n, double* Linv_out) {
  BASQ_CHECK(A && Linv_out && n >= 1, BASQ_ERR_INVALID, "spd_inverse_factor: bad argument");
  OrthWs ws;
  BASQ_TRY(ws.alloc(ctx, n, 0));
  BASQ_CUDA(cudaMemcpyAsync(ws.gram.p, A, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToDevice, ctx->stream));
  BASQ_TRY(chol_inverse(ctx, ws, n, 1e-300));
  BASQ_CUDA(cudaMemcpyAsync(Linv_out, ws.linv.p, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToDevice, ctx->stream));
  return ws.check_status(ctx, "spd_inverse_factor");
}

namespace {
// The diagonal block A [b, b] (ld lda) made symmetric from its lower triangle, in place, and copied to dst (ld b)
__global__ void sym_block_kernel(double* __restrict__ A, int64_t lda, int b, double* __restrict__ dst) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= b * b) return;
  const int i = t / b, j = t % b;
  const double v = i >= j ? A[(int64_t)i * lda + j] : A[(int64_t)j * lda + i];
  if (i < j) A[(int64_t)i * lda + j] = v;
  dst[t] = v;
}
}  // namespace

// In place: the lower triangle of the symmetric positive definite A [n, n] (row-major, ld n; only the lower
// triangle is read) becomes its Cholesky factor G, A = G G^T.  The upper triangle is left with scratch values.
// Blocked right-looking, panels of 256 columns:
//   - the diagonal block goes through the cooperative Cholesky + inverse kernel above (G_kk^-1);
//   - the column panel, diagonal block included, is A[k:, k:k+b] G_kk^-T (A_kk G_kk^-T = G_kk): one DMMA GEMM
//     against a lower-triangular operand;
//   - the trailing matrix loses P P^T of the panel rows below the diagonal block, lower tiles only.
// n^3 / 3 flop, nearly all of it in the trailing updates; no triangular inverse of the whole matrix.
int spd_chol_blocked(basq_ctx* ctx, double* A, int n) {
  constexpr int CHB = 256;
  BASQ_CHECK(A && n >= 1, BASQ_ERR_INVALID, "spd_chol_blocked: bad argument");
  const int nb = n < CHB ? n : CHB;
  OrthWs ws;
  DevBuf panel;
  BASQ_TRY(ws.alloc(ctx, nb, 0));
  BASQ_TRY(panel.alloc(ctx, sizeof(double) * (size_t)n * CHB));
  for (int k = 0; k < n; k += CHB) {
    const int b = std::min(CHB, n - k);
    double* Akk = A + (int64_t)k * n + k;
    sym_block_kernel<<<ceil_div(b * b, 256), 256, 0, ctx->stream>>>(Akk, n, b, ws.gram.as<double>());
    ctx->launches++;
    BASQ_TRY(chol_inverse(ctx, ws, b, 1e-300));
    // P [n - k, b] (ld CHB) = A[k:, k:k+b] G_kk^-T, written back over the panel's columns
    BASQ_TRY(dgemm(ctx, false, true, n - k, b, b, 1.0, Akk, n, ws.linv.as<double>(), b, 0.0, panel.as<double>(), CHB,
                   /*b_lower_tri=*/true));
    BASQ_CUDA(cudaMemcpy2DAsync(Akk, sizeof(double) * n, panel.p, sizeof(double) * CHB, sizeof(double) * b, n - k,
                                cudaMemcpyDeviceToDevice, ctx->stream));
    const int t = n - k - b;
    if (t > 0) {
      const double* Pb = panel.as<double>() + (int64_t)b * CHB;
      BASQ_TRY(dgemm(ctx, false, true, t, t, b, -1.0, Pb, CHB, Pb, CHB, 1.0, Akk + (int64_t)b * n + b, n, false, false,
                     false, /*c_lower_only=*/true));
    }
  }
  return ws.check_status(ctx, "spd_chol_blocked");
}

// Rank r of `world` (shard == nullptr: one rank holding everything) owns rows [r chunk, min(M, (r + 1) chunk)),
// chunk = ceil(M / world), of K(Z, Z) - it evaluates, converts and multiplies only those.  Sharded (multi-GPU), the
// ranks meet twice per product: a sum of the q x q Gram matrices (CholeskyQR) and an all-gather of the
// orthonormalised rows, both done by the caller's exchange function on buffers the caller owns (the library stays
// free of any communication dependency; basq_b200/sharded.py passes torch.distributed collectives).  rows_buf
// [world * chunk, q] is the full basis in global row order (rank r's rows at r * chunk).  The Cholesky
// factorisations are replicated, so every rank takes the same decisions and issues the same exchanges.
int nystrom_basis(basq_ctx* ctx, const basq_kernel_desc* desc, const void* Z, int64_t M, int q, const double* Omega,
                  int niter, double* U_out, double* S_out, const NysShard* shard) {
  PhaseTimer timer(ctx, PH_NYS);
  BASQ_CHECK(q >= 1 && q <= M, BASQ_ERR_INVALID, "nystrom: need 1 <= q <= M (q=%d M=%lld)", q, (long long)M);
  const int rank = shard ? shard->rank : 0, world = shard ? shard->world : 1;
  BASQ_CHECK(!shard || (world >= 1 && rank >= 0 && rank < world && shard->fn && shard->gram_buf && shard->rows_buf &&
                        !S_out),
             BASQ_ERR_INVALID, "nystrom (sharded): bad rank / world / buffers");
  BASQ_CHECK(M <= 46000 * (int64_t)world, BASQ_ERR_UNSUPPORTED, "nystrom: M=%lld landmarks need a %.1f GB Gram matrix%s",
             (long long)M, 8.0 * M * M / world / 1e9, shard ? " per rank" : "");
  BASQ_CHECK(niter >= 0 && niter <= 16, BASQ_ERR_INVALID, "nystrom: niter out of range");
  const int64_t chunk = (M + world - 1) / world;
  const int64_t row0 = std::min<int64_t>(M, (int64_t)rank * chunk);
  const int nr = (int)(std::min<int64_t>(M, row0 + chunk) - row0);
  const int Mi = (int)M;
  const size_t esz = desc->dtype == BASQ_F64 ? 8 : 4;
  DevBuf K, Y, Y2, drawn;
  if (!Omega) {
    // torch.svd_lowrank draws its own Gaussian test matrix (BASQ/_rchq.py:28-31); so does the library when
    // the caller passes none: Philox stream of key seed + number of earlier draws (basq_ctx_set_seed), the
    // same on every rank
    BASQ_TRY(drawn.alloc(ctx, sizeof(double) * (size_t)M * q));
    BASQ_TRY(standard_normals(ctx, ctx->seed + ctx->draws, 0, M, q, drawn.as<double>()));
    ctx->draws++;
    Omega = drawn.as<double>();
  }
  BASQ_TRY(K.alloc(ctx, sizeof(double) * (size_t)std::max(nr, 1) * M));
  BASQ_TRY(Y.alloc(ctx, sizeof(double) * (size_t)std::max(nr, 1) * q));
  if (!shard) BASQ_TRY(Y2.alloc(ctx, sizeof(double) * (size_t)M * q));
  OrthWs ws;
  BASQ_TRY(ws.alloc(ctx, q, std::max(nr, 1)));
  // K [nr, M] = K(Z, Z)[rows, :].  fp32 kernels: products on the tensor cores (fp16 hi/lo split products, tgemm.cu) -
  // the Gram matrix itself is only fp32-accurate, and the subspace iteration re-orthonormalises in fp64 after every
  // product; fp64 kernels: fp64 GEMM.  K(Z, Z) is symmetric, so K^T Y = K Y.
  const bool tensor = desc->dtype == BASQ_F32;
  BlkOperand Kb, Yb;
  if (nr > 0) {
    const unsigned char* Zr = static_cast<const unsigned char*>(Z) + (size_t)row0 * desc->d * esz;
    BASQ_TRY(gram_matrix(ctx, desc, Zr, nr, Z, M, K.as<double>(), tensor, /*diag_col0=*/row0));
    if (tensor) {
      BASQ_TRY(Kb.alloc(ctx, nr, Mi));
      BASQ_TRY(blk_from_f64(ctx, K.as<double>(), M, false, &Kb));
      BASQ_TRY(Yb.alloc(ctx, q, Mi));
    }
  }
  double* Yr = Y.as<double>();                                  // [nr, q] this rank's rows of the latest product
  double* Yfull = shard ? shard->rows_buf : Y2.as<double>();    // [M, q] the input of the next product
  // Yr <- K[rows, :] Yin  (Yin: a full [M, q] matrix)
  auto multiply = [&](const double* Yin) -> int {
    if (nr == 0) return BASQ_OK;
    if (!tensor) return dgemm(ctx, false, false, nr, q, Mi, 1.0, K.as<double>(), M, Yin, q, 0.0, Yr, q);
    BASQ_TRY(blk_from_f64(ctx, Yin, q, true, &Yb));                 // Y^T as [q, M] operand
    return tgemm(ctx, Yb, Kb, 1.0, Yr, q, true);                    // (Y^T K^T)^T = K Y
  };
  // Yfull <- every rank's Yr.  One rank: the two buffers trade roles (no copy), the next product writes the other.
  auto publish = [&]() -> int {
    if (!shard) {
      std::swap(Yr, Yfull);
      return BASQ_OK;
    }
    if (nr > 0)
      BASQ_CUDA(cudaMemcpyAsync(Yfull + (size_t)row0 * q, Yr, sizeof(double) * (size_t)nr * q, cudaMemcpyDeviceToDevice,
                                ctx->stream));
    BASQ_CHECK(shard->fn(shard->user, BASQ_XCHG_ALLGATHER_ROWS, chunk * q) == 0, BASQ_ERR_INVALID,
               "nystrom: the exchange function failed (all-gather of the basis rows)");
    return BASQ_OK;
  };
  // Between products one shifted CholeskyQR pass is enough: it only has to keep the basis well
  // enough conditioned for the next product (directions it damps by more than the working precision
  // are lost to that product's rounding anyway); the last product is followed by passes until the
  // basis is orthonormal to fp64 (two at M = 1e4, q = 999, d = 10: |U U^T - I| = 9e-15; three for
  // numerically rank-deficient Gram matrices such as d = 2).
  constexpr int TO_FP64 = -1;   // orthonormalise's adaptive passes
  BASQ_TRY(multiply(Omega));
  BASQ_TRY(orthonormalise(ctx, ws, Yr, nr, q, niter > 0 ? 1 : TO_FP64, M, shard));
  BASQ_TRY(publish());
  // Within a power iteration (K^T then K) the intermediate basis need not be re-orthonormalised when
  // the spectrum behind the basis is flat enough: two products damp the weakest captured direction by
  // (sigma_q / sigma_1)^2 relative to the strongest, which must stay well above the split product's rounding
  // (1e-7) of the second product.  sigma_q / sigma_1 is read off the diagonal of the Cholesky factor
  // of the first CholeskyQR pass (L^-1 is at hand, and replicated: every rank takes the same decision).
  // Measured at M = 1e4, q = 999, d = 10 (spread 0.38): the captured trace tr(U K U^T) agrees to 9 digits
  // with the fully re-orthonormalised run (1530.730019 vs 1530.730022); at d = 2 (spread 1e-8) the skip
  // would double the approximation error, and the criterion keeps every orthonormalisation.
  // BASQ_NYS_ORTH_MID=1 forces them all.
  const bool force_mid = [] { const char* e = getenv("BASQ_NYS_ORTH_MID"); return e && e[0] == '1'; }();  // read per call (tests toggle it)
  bool skip_mid = false;
  if (!force_mid && niter > 0) {
    diag_spread_kernel<<<1, 256, 0, ctx->stream>>>(ws.linv.as<double>(), q, q, ws.scal.as<double>());
    ctx->launches++;
    double spread = 0.0;  // of diag(L^-1) = 1 / diag(L): the same ratio
    BASQ_CUDA(cudaMemcpyAsync(&spread, ws.scal.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
    skip_mid = spread > 1e-2;
    if (ctx->trace) fprintf(stderr, "[nystrom] singular-value spread of K Omega ~ %.3g -> %s\n", spread,
                            skip_mid ? "one orthonormalisation per power iteration" : "orthonormalise after every product");
  }
  for (int it = 0; it < niter; ++it) {
    BASQ_TRY(multiply(Yfull));
    if (!skip_mid) BASQ_TRY(orthonormalise(ctx, ws, Yr, nr, q, 1, M, shard));
    BASQ_TRY(publish());
    BASQ_TRY(multiply(Yfull));
    BASQ_TRY(orthonormalise(ctx, ws, Yr, nr, q, it + 1 == niter ? TO_FP64 : 1, M, shard));
    BASQ_TRY(publish());
  }
  // U = Q^T  [q, M]
  {
    dim3 grid((unsigned)ceil_div(q, 32), (unsigned)ceil_div(Mi, 32));
    transpose_kernel<<<grid, dim3(32, 8), 0, ctx->stream>>>(Yfull, Mi, q, U_out);
    ctx->launches++;
  }
  if (S_out) {
    // Rayleigh quotients q_i^T K q_i (one rank: K holds every row; Yr is free scratch)
    BASQ_TRY(dgemm(ctx, false, false, Mi, q, Mi, 1.0, K.as<double>(), M, Yfull, q, 0.0, Yr, q));
    BASQ_TRY(dgemm(ctx, true, false, q, q, Mi, 1.0, Yfull, q, Yr, q, 0.0, ws.gram.as<double>(), q));
    diag_kernel<<<ceil_div(q, 256), 256, 0, ctx->stream>>>(ws.gram.as<double>(), q, q, S_out);
    ctx->launches++;
  }
  BASQ_CUDA(cudaGetLastError());
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

}  // namespace basq
