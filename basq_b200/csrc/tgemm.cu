// Dense fp32-accuracy GEMM on the 5th-generation tensor cores (fp16 hi / lo split, fp32 accumulate in TMEM):
//
//   D[I, J] = A[I, Kd] * B[J, Kd]^T
//
// used for the Nystrom subspace iteration (K(Z,Z) Y, reference torch.svd_lowrank inside
// ker_svd_sparsify, BASQ/_rchq.py:28-31) and the posterior-covariance Gram correction
// (K_ZX W K_Xy, BASQ/_gp.py:259-277) when the kernel is evaluated in fp32.
//
// Operands are stored "row-scaled + blocked + split" (BlkOperand): every row is multiplied by a power of two
// that brings its largest magnitude into [2^13, 2^14), then x = hi + lo with hi = fp16(x), lo = fp16(x - hi)
// (22 significant bits, the same as a 2 x TF32 split at half the bytes and twice the MMA rate), laid out
// [row tile of 128][K chunk of 8][128 rows][8] so that one (row tile, 64-wide K block) is a contiguous 16 KB
// piece that a single bulk copy (cp.async.bulk, UBLKCP) drops into shared memory in exactly the K-major
// no-swizzle form the tcgen05 shared-memory descriptor expects (8-row core matrices contiguous, SBO = 128 B,
// LBO = 128 rows * 16 B).  Three MMAs per K step (lo*hi, hi*lo, hi*hi; kind::f16, M = 128, N = 128, K = 16)
// reproduce the fp32 product to ~2^-21; the epilogue undoes the two row scales (exact).
//
// CTA = 6 warps, persistent, one CTA per SM; tile 128 x 256 (two 128-column accumulators):
//   warp 0    producer: six 8 KB bulk copies per 32-wide K block (A hi/lo, B0 hi/lo, B1 hi/lo), 4-stage ring
//   warp 1    TMEM allocation + tcgen05.mma issue (12 MMAs per K block, one lane)
//   warps 2-5 epilogue: tcgen05.ld -> fp64 store (plain or transposed); double-buffered accumulators
//             (2 x 256 TMEM columns) so the epilogue of one tile overlaps the main loop of the next
// Work split.  One unit = (tile, K part); units are dealt round-robin to the persistent CTAs in K-part-major order
// (SegWalk).  With one K part per tile, 320 tiles on 148 SMs take 3 rounds for 2.16 rounds of work; with two
// parts, 5 half rounds.
#include <math_constants.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "setsum_mma.cuh"  // mma:: helpers (mbarrier, bulk copy, tcgen05 wrappers, smem descriptor)
#include "tgemm.cuh"

namespace basq {

namespace {

constexpr int TG_THREADS = 192;
// K block = TG_KCH chunks of 8 (one bulk copy per operand piece); deeper ring of smaller stages keeps more copies in
// flight: the kernel is bound by the operand stream (A/B: -DBASQ_TG_KCH=8 -DBASQ_TG_NSTAGE=2 was round 1's shape)
#ifndef BASQ_TG_KCH
#define BASQ_TG_KCH 4
#endif
#ifndef BASQ_TG_NSTAGE
#define BASQ_TG_NSTAGE 4
#endif
constexpr int TG_KCH = BASQ_TG_KCH;
constexpr int TG_NSTAGE = BASQ_TG_NSTAGE;
constexpr int TG_PIECE = TG_KCH * 128 * 16;       // bytes of one (row tile, K block) piece
constexpr int TG_STAGE_BYTES = 6 * TG_PIECE;      // A hi, A lo, B0 hi, B0 lo, B1 hi, B1 lo
constexpr int TG_SMEM = TG_NSTAGE * TG_STAGE_BYTES + 256;

struct TgDev {
  const __half *Ahi, *Alo, *Bhi, *Blo;
  const float *Ainv, *Binv;  // 1 / row scale
  int I, J;        // logical output size
  int RT_A, RT_B;  // row tiles
  int KC;          // K chunks (of 8) = 8 * K blocks
  double* out;
  int64_t ldo;
  int transposed;  // 0: out[i * ldo + j] ; 1: out[j * ldo + i]
  double alpha;
  int accumulate;  // out += alpha * A B^T instead of out = ...
  int ksplit;      // 1 or 2 K parts per tile (2: both parts are added onto the zero-filled / accumulated-into output)
};

// The segments (tile, K blocks [kb_lo, kb_hi)) of this CTA, in order.  All three roles walk the same list.
// Units are numbered K-part major (all tiles of the first K part, then all tiles of the second) and dealt out
// round-robin, so the CTAs that run together stream the same K blocks at the same time: the pieces they share
// (a B tile pair is read by RT_A CTAs, an A tile by all tile columns) meet in L2.
struct SegWalk {
  int cur, end, n_items, nkb, step, parts;
  __device__ SegWalk(const TgDev& a, int n_items_, int nkb_)
      : cur((int)blockIdx.x), end(n_items_ * a.ksplit), n_items(n_items_), nkb(nkb_), step((int)gridDim.x), parts(a.ksplit) {}
  __device__ bool next(int& item, int& kb_lo, int& kb_hi) {
    if (cur >= end) return false;
    const int part = cur / n_items;
    item = cur - part * n_items;
    kb_lo = (int)((int64_t)nkb * part / parts);
    kb_hi = (int)((int64_t)nkb * (part + 1) / parts);
    cur += step;
    return true;
  }
};

__global__ void __launch_bounds__(TG_THREADS, 1) tgemm_kernel(const TgDev a) {
  extern __shared__ __align__(1024) unsigned char smem_tg[];
  unsigned char* const smem = smem_tg;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TG_NSTAGE * TG_STAGE_BYTES);
  uint64_t* s_full = bars;                    // [NSTAGE]
  uint64_t* s_empty = bars + TG_NSTAGE;       // [NSTAGE]
  uint64_t* t_full = bars + 2 * TG_NSTAGE;    // [2]
  uint64_t* t_empty = t_full + 2;             // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < TG_NSTAGE; ++s) {
      mma::mbar_init(&s_full[s], 1);
      mma::mbar_init(&s_empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mma::mbar_init(&t_full[b], 1);
      mma::mbar_init(&t_empty[b], 4);
    }
    mma::fence_barrier_init();
  }
  if (warp == 1) mma::tmem_alloc(tmem_slot, 512);
  mma::tc_fence_before();
  __syncthreads();
  mma::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_tb = (a.RT_B + 1) / 2;
  const int n_items = a.RT_A * n_tb;
  const int nkb = a.KC / TG_KCH;
  const size_t tile_el = (size_t)a.KC * 128 * 8;  // halves per row tile

  if (warp == 0) {
    // ======================================================================== producer
    if (lane == 0) {
      uint32_t it = 0;
      SegWalk walk(a, n_items, nkb);
      int item, kb_lo, kb_hi;
      while (walk.next(item, kb_lo, kb_hi)) {
        const int ta = item % a.RT_A, tb = item / a.RT_A;
        const int tb0 = 2 * tb, tb1 = min(2 * tb + 1, a.RT_B - 1);  // an odd tail re-reads the last tile (discarded)
        for (int kb = kb_lo; kb < kb_hi; ++kb, ++it) {
          const int s = it % TG_NSTAGE;
          mma::mbar_wait(&s_empty[s], ((it / TG_NSTAGE) & 1u) ^ 1u);
          unsigned char* st = smem + (size_t)s * TG_STAGE_BYTES;
          mma::mbar_expect_tx(&s_full[s], TG_STAGE_BYTES);
          const size_t koff = (size_t)kb * TG_KCH * 128 * 8;
          mma::bulk_g2s(st + 0 * TG_PIECE, a.Ahi + ta * tile_el + koff, TG_PIECE, &s_full[s]);
          mma::bulk_g2s(st + 1 * TG_PIECE, a.Alo + ta * tile_el + koff, TG_PIECE, &s_full[s]);
          mma::bulk_g2s(st + 2 * TG_PIECE, a.Bhi + tb0 * tile_el + koff, TG_PIECE, &s_full[s]);
          mma::bulk_g2s(st + 3 * TG_PIECE, a.Blo + tb0 * tile_el + koff, TG_PIECE, &s_full[s]);
          mma::bulk_g2s(st + 4 * TG_PIECE, a.Bhi + tb1 * tile_el + koff, TG_PIECE, &s_full[s]);
          mma::bulk_g2s(st + 5 * TG_PIECE, a.Blo + tb1 * tile_el + koff, TG_PIECE, &s_full[s]);
        }
      }
    }
  } else if (warp == 1) {
    // ======================================================================== MMA issuer
    // kind::f16: fp16 operands (format 0), fp32 accumulator, N = 128, M = 128
    constexpr uint32_t IDESC = (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(128 >> 3) << 17) | ((128u >> 4) << 24);
    uint32_t it = 0, tc = 0;
    SegWalk walk(a, n_items, nkb);
    int item, kb_lo, kb_hi;
    for (; walk.next(item, kb_lo, kb_hi); ++tc) {
      const uint32_t buf = tc & 1u;
      mma::mbar_wait(&t_empty[buf], ((tc >> 1) & 1u) ^ 1u);
      mma::tc_fence_after();
      for (int kb = kb_lo; kb < kb_hi; ++kb, ++it) {
        const int s = it % TG_NSTAGE;
        mma::mbar_wait(&s_full[s], (it / TG_NSTAGE) & 1u);
        mma::tc_fence_after();
        if (lane == 0) {
          const uint32_t st = mma::smem_u32(smem + (size_t)s * TG_STAGE_BYTES);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t d = tmem_base + buf * 256 + h * 128;
            const uint32_t ahi = st, alo = st + TG_PIECE;
            const uint32_t bhi = st + (2 + 2 * h) * TG_PIECE, blo = bhi + TG_PIECE;
#pragma unroll
            for (int p = 0; p < 3; ++p) {
              const uint32_t aa = (p == 0) ? alo : ahi;   // lo*hi, hi*lo, hi*hi
              const uint32_t bb = (p == 1) ? blo : bhi;
#pragma unroll
              for (int ks = 0; ks < TG_KCH / 2; ++ks) {
                const uint64_t ad = mma::smem_desc(aa + ks * 2 * (128 * 16), 128 * 16, 128);
                const uint64_t bd = mma::smem_desc(bb + ks * 2 * (128 * 16), 128 * 16, 128);
                mma::umma_f16(d, ad, bd, IDESC, (kb > kb_lo || p > 0 || ks > 0) ? 1u : 0u);
              }
            }
          }
          mma::umma_commit(&s_empty[s]);
          if (kb == kb_hi - 1) mma::umma_commit(&t_full[buf]);
        }
        __syncwarp();
      }
    }
  } else {
    // ======================================================================== epilogue
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    uint32_t tc = 0;
    SegWalk walk(a, n_items, nkb);
    int item, kb_lo, kb_hi;
    for (; walk.next(item, kb_lo, kb_hi); ++tc) {
      const int ta = item % a.RT_A, tb = item / a.RT_A;
      const uint32_t buf = tc & 1u;
      const bool partial = (kb_hi - kb_lo) != nkb;   // the other K part of this tile is another unit
      mma::mbar_wait(&t_full[buf], (tc >> 1) & 1u);
      mma::tc_fence_after();
      const int i = ta * 128 + row;
      const double ai = (i < a.I) ? a.alpha * (double)a.Ainv[i] : 0.0;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * 256;
      const int ncols = min(256, a.J - tb * 256);  // an odd tail's second half lies beyond J
#pragma unroll 1
      for (int cb = 0; cb < ncols; cb += 32) {
        uint32_t v[32];
        mma::tmem_ld32(taddr + cb, v);
        mma::tmem_ld_wait();
        if (i < a.I) {
          const int j0 = tb * 256 + cb;
#pragma unroll
          for (int c = 0; c < 32; ++c)
            if (j0 + c < a.J) {
              double* dst = a.transposed ? a.out + (int64_t)(j0 + c) * a.ldo + i : a.out + (int64_t)i * a.ldo + j0 + c;
              const double val = ai * (double)a.Binv[j0 + c] * (double)__uint_as_float(v[c]);
              if (partial) atomicAdd(dst, val);
              else *dst = a.accumulate ? *dst + val : val;
            }
        }
      }
      mma::tc_fence_before();
      __syncwarp();
      if (lane == 0) mma::mbar_arrive(&t_empty[buf]);
    }
  }

  mma::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    mma::tc_fence_after();
    mma::tmem_dealloc(tmem_base, 512);
  }
}

// Row scale of operand row `row`: 2^(13 - floor(log2 max_k |x|)), its inverse in rinv; rows beyond `rows` get 0.
__device__ __forceinline__ void write_rowscale(double mx, bool valid, float* rscale, float* rinv, int row) {
  float r = 0.f, iv = 0.f;
  if (valid) {
    int e = 0;
    if (mx > 0.0 && isfinite(mx)) e = 13 - ilogb(mx);
    e = max(-100, min(100, e));
    r = ldexpf(1.f, e);
    iv = ldexpf(1.f, -e);
  }
  rscale[row] = r;
  rinv[row] = iv;
}

// src [rows, kdim]: one block per operand row
__global__ void blk_rowscale_kernel(const double* __restrict__ src, int64_t ld, int rows, int kdim, float* __restrict__ rscale,
                                    float* __restrict__ rinv) {
  __shared__ double sh[256];
  const int row = blockIdx.x;
  double mx = 0.0;
  if (row < rows)
    for (int k = threadIdx.x; k < kdim; k += 256) mx = fmax(mx, fabs(src[(int64_t)row * ld + k]));
  sh[threadIdx.x] = mx;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + w]);
    __syncthreads();
  }
  if (threadIdx.x == 0) write_rowscale(sh[0], row < rows, rscale, rinv, row);
}

// src [kdim, rows] (the operand is src^T): a block of 32 x 8 threads covers 32 operand rows (columns of src) and
// one slice of k; the slices meet in mx[] through an integer max (non-negative doubles order like their bits)
__global__ void blk_rowmax_t_kernel(const double* __restrict__ src, int64_t ld, int rows, int kdim, int kslice,
                                    unsigned long long* __restrict__ mx_bits) {
  __shared__ double sh[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int row = blockIdx.x * 32 + tx;
  const int k0 = blockIdx.y * kslice, k1 = min(kdim, k0 + kslice);
  double mx = 0.0;
  if (row < rows)
    for (int k = k0 + ty; k < k1; k += 8) mx = fmax(mx, fabs(src[(int64_t)k * ld + row]));
  sh[ty][tx] = mx;
  __syncthreads();
  if (ty == 0 && row < rows) {
    for (int y = 1; y < 8; ++y) mx = fmax(mx, sh[y][tx]);
    if (!(mx == mx)) mx = CUDART_INF;   // a NaN entry: keep the scale at 1 (write_rowscale), the product carries the NaN
    atomicMax(&mx_bits[row], (unsigned long long)__double_as_longlong(mx));
  }
}
__global__ void blk_rowscale_finish_kernel(const unsigned long long* __restrict__ mx_bits, int rows, int padded,
                                           float* __restrict__ rscale, float* __restrict__ rinv) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= padded) return;
  write_rowscale(row < rows ? __longlong_as_double((long long)mx_bits[row]) : 0.0, row < rows, rscale, rinv, row);
}

// one thread per (row tile, chunk, row): 8 consecutive K elements of one operand row
template <bool TRANSPOSED>
__global__ void blk_split_kernel(const double* __restrict__ src, int64_t ld, int rows, int kdim, int RT, int KC,
                                 const float* __restrict__ rscale, __half* __restrict__ hi, __half* __restrict__ lo) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)RT * KC * 128;
  if (t >= total) return;
  const int r = (int)(t % 128);
  const int kc = (int)((t / 128) % KC);
  const int rt = (int)(t / (128 * (int64_t)KC));
  const int row = rt * 128 + r;
  const double rs = row < rows ? (double)rscale[row] : 0.0;
  __half h[8], l[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = kc * 8 + e;
    double x = 0.0;
    if (row < rows && k < kdim) x = (TRANSPOSED ? src[(int64_t)k * ld + row] : src[(int64_t)row * ld + k]) * rs;
    h[e] = __double2half(x);
    // the residual is taken against the fp64 value: hi + lo carries ~22 bits of x
    l[e] = __double2half(x - (double)__half2float(h[e]));
  }
  reinterpret_cast<uint4*>(hi)[t] = *reinterpret_cast<const uint4*>(h);
  reinterpret_cast<uint4*>(lo)[t] = *reinterpret_cast<const uint4*>(l);
}

}  // namespace

int BlkOperand::alloc(basq_ctx* ctx, int rows_, int kdim_) {
  rows = rows_;
  kdim = kdim_;
  RT = ceil_div(rows_, 128);
  KC = ceil_div(kdim_, 64) * 8;
  const size_t bytes = sizeof(__half) * (size_t)RT * KC * 128 * 8;
  BASQ_TRY(hi.alloc(ctx, bytes));
  BASQ_TRY(lo.alloc(ctx, bytes));
  BASQ_TRY(rinv.alloc(ctx, sizeof(float) * (size_t)RT * 128));
  return BASQ_OK;
}

int blk_from_f64(basq_ctx* ctx, const double* src, int64_t ld, bool transposed, BlkOperand* op) {
  const int padded = op->RT * 128;
  DevBuf rscale;
  BASQ_TRY(rscale.alloc(ctx, sizeof(float) * (size_t)padded));
  DevBuf mx;
  if (transposed) {
    BASQ_TRY(mx.alloc(ctx, sizeof(unsigned long long) * (size_t)padded));
    BASQ_CUDA(cudaMemsetAsync(mx.p, 0, sizeof(unsigned long long) * (size_t)padded, ctx->stream));
    const int slices = std::max(1, std::min(64, op->kdim / 128));
    const int kslice = ceil_div(op->kdim, slices);
    blk_rowmax_t_kernel<<<dim3((unsigned)ceil_div(padded, 32), (unsigned)ceil_div(op->kdim, kslice)), 256, 0, ctx->stream>>>(
        src, ld, op->rows, op->kdim, kslice, mx.as<unsigned long long>());
    blk_rowscale_finish_kernel<<<ceil_div(padded, 256), 256, 0, ctx->stream>>>(mx.as<unsigned long long>(), op->rows, padded,
                                                                              rscale.as<float>(), op->rinv.as<float>());
    ctx->launches++;
  } else {
    blk_rowscale_kernel<<<padded, 256, 0, ctx->stream>>>(src, ld, op->rows, op->kdim, rscale.as<float>(),
                                                         op->rinv.as<float>());
  }
  const int64_t total = (int64_t)op->RT * op->KC * 128;
  const unsigned grid = (unsigned)ceil_div64(total, 256);
  if (transposed)
    blk_split_kernel<true><<<grid, 256, 0, ctx->stream>>>(src, ld, op->rows, op->kdim, op->RT, op->KC, rscale.as<float>(),
                                                          op->hi.as<__half>(), op->lo.as<__half>());
  else
    blk_split_kernel<false><<<grid, 256, 0, ctx->stream>>>(src, ld, op->rows, op->kdim, op->RT, op->KC, rscale.as<float>(),
                                                           op->hi.as<__half>(), op->lo.as<__half>());
  ctx->launches += 2;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;   // `rscale` returns to the context's block cache; stream order keeps it intact until the split kernel has run
}

int tgemm(basq_ctx* ctx, const BlkOperand& A, const BlkOperand& B, double alpha, double* out, int64_t ldo,
          bool transposed, bool accumulate) {
  BASQ_CHECK(A.kdim == B.kdim && A.KC == B.KC, BASQ_ERR_INVALID, "tgemm: inner dimensions differ (%d vs %d)", A.kdim,
             B.kdim);
  BASQ_CHECK((size_t)TG_SMEM <= ctx->smem_optin, BASQ_ERR_UNSUPPORTED, "tgemm: needs %d B shared memory", TG_SMEM);
  if (A.rows <= 0 || B.rows <= 0) return BASQ_OK;
  TgDev d;
  d.Ahi = A.hi.as<__half>(); d.Alo = A.lo.as<__half>();
  d.Bhi = B.hi.as<__half>(); d.Blo = B.lo.as<__half>();
  d.Ainv = A.rinv.as<float>(); d.Binv = B.rinv.as<float>();
  d.I = A.rows; d.J = B.rows;
  d.RT_A = A.RT; d.RT_B = B.RT;
  d.KC = A.KC;
  d.out = out; d.ldo = ldo;
  d.transposed = transposed ? 1 : 0;
  d.alpha = alpha;
  d.accumulate = accumulate ? 1 : 0;
  const int n_items = A.RT * ((B.RT + 1) / 2);
  const int grid = std::min(ctx->num_sms, n_items);
  // Two K parts per tile when that needs fewer rounds of the grid (320 tiles on 148 SMs: 3 rounds whole, 5 half
  // rounds split).  Two addends per element: the sum does not depend on their order.  (Cutting the (tile, K block)
  // sequence into equal contiguous ranges - "stream-K" - balances perfectly but lets neighbouring CTAs drift
  // apart in K: measured L2 hit rate 20 % instead of 76 %, 3.8 GB instead of 0.54 GB from HBM, and slower.)
  const int nkb = A.KC / TG_KCH;
  d.ksplit = 1;
  if (nkb >= 8 && 2 * ceil_div(n_items, grid) > ceil_div(2 * n_items, grid)) d.ksplit = 2;
  if (d.ksplit > 1 && !accumulate) {   // both parts are added onto zeros
    const size_t width = sizeof(double) * (size_t)(transposed ? d.I : d.J);
    BASQ_CUDA(cudaMemset2DAsync(out, sizeof(double) * (size_t)ldo, 0, width, (size_t)(transposed ? d.J : d.I), ctx->stream));
  }
  BASQ_CUDA(cudaFuncSetAttribute(tgemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TG_SMEM));
  tgemm_kernel<<<grid, TG_THREADS, TG_SMEM, ctx->stream>>>(d);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

}  // namespace basq
