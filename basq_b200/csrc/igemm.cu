// fp64 matrix product on the 5th-generation tensor cores with int8 digits (Ozaki slicing):
//
//   C[i, j] (+)= alpha * sum_k A[i, k] B[j, k]
//
// used for the projection of the level columns, rows 1..q of U' Gf (session_level_project), where it replaces
// the fp64 DMMA GEMM: the int8 pipe does about 100x the fp64 tensor rate and the digit products are exact.
//
// Slicing (dig_from_f64).  Every row of A and every column of the product (row j of B) gets a power of two 2^e,
// e = E - 6 with E the frexp exponent of the row's largest magnitude, so that y = x 2^-e lies in (-64, 64); then
// d_0 = rint(y), y <- 128 (y - d_0), d_1 = rint(y), ... - every step exact in fp64, |d_a| <= 64 - gives
//   x = 2^e (sum_{a<8} d_a 2^(-7a) + r),  |r| <= 2^-50,  i.e. |x - sliced x| <= 2^-55 max_k |x_row|.
// Eight digits cover the 53 bits of the row's largest entries; smaller entries keep the bits above 2^-55 of it.
//
// Products.  Digit pairs (a, b) with a + b <= 7 (36 int8 GEMMs), all pairs of one diagonal t = a + b (weight
// 2^(-7t)) into one s32 TMEM accumulator.  A diagonal holds at most 8 pairs of products of magnitude <= 64^2,
// so its sum is exact while 8 * Kc * 2^12 < 2^31: K is cut into launches of at most IG_KMAX_BLOCKS blocks
// (65504 elements) whose results are added in fp64.
//
// Combine.  Each diagonal's s32 sum converts to fp64 exactly; Horner from the smallest weight up,
// acc = D_7; acc = acc 2^-7 + D_t, adds them (only these 7 additions round), then ldexp undoes the two scales.
//
// Error bound.  With a_i = max_k |A[i, k]|, b_j = max_k |B[j, k]| (both scaled entries lie in [32, 64) at the max),
// per k the dropped diagonals t >= 8 contribute at most 2^12 sum_{t>=8} (15 - t) 2^(-7t) < 7.1 2^-44 and the
// two residuals at most 2 * 64 * 2^-50 in scaled units, against a scaled a_i b_j >= 2^10:
//   |C - C~| <= 2^-50.8 K a_i b_j + 7 u |C~|     (u = 2^-53)
// The first term is absolute in the row and column maxima: entries far below their row's (column's) maximum keep
// fewer of their own bits than fp64 arithmetic would give them.  The projection's operands (rows of U', columns
// of folded set sums) lie within a few decades of their maxima, where the error is at the level of fp64 rounding
// (tests/test_gpu_igemm.py).
//
// CTA = 6 warps, one 128 x 64 output tile per CTA (grid = column tiles x row tiles):
//   warp 0    producer: one bulk copy of the A piece (8 digits x 128 rows x 32 K, 32 KB) and one of the B piece
//             (8 x 64 x 32, 16 KB) per K block, 4-stage ring
//   warp 1    TMEM allocation (8 diagonals x 64 columns = all 512) + tcgen05.mma kind::i8 issue: the 36 digit
//             products of a K block as 12 MMAs, each A digit against up to 4 B digits stacked along N (shared
//             memory reads per K block 120 KB instead of 216 KB for 36 MMAs of N = 64)
//   warps 2-5 epilogue: tcgen05.ld of the 8 diagonals -> fp64 combine -> store
#include <math_constants.h>

#include <algorithm>

#include "common.cuh"
#include "igemm.cuh"
#include "setsum_mma.cuh"  // mma:: helpers (mbarrier, bulk copy, tcgen05 wrappers, smem descriptor)

namespace basq {

namespace {

constexpr int IG_BM = 128, IG_BN = 64;
constexpr int IG_NDIAG = IG_DIGITS;                            // diagonals t = a + b <= IG_DIGITS - 1
constexpr int IG_A_BYTES = IG_DIGITS * IG_KB * IG_BM;           // 32 KB: one (row tile, K block) piece of A
constexpr int IG_B_BYTES = IG_DIGITS * IG_KB * IG_BN;           // 16 KB
constexpr int IG_STAGE_BYTES = IG_A_BYTES + IG_B_BYTES;
constexpr int IG_NSTAGE = 4;
constexpr int IG_SMEM = IG_NSTAGE * IG_STAGE_BYTES + 256;
constexpr int IG_THREADS = 192;
constexpr int IG_KMAX_BLOCKS = 2047;                            // 8 pairs * 2047 * 32 * 64^2 < 2^31
static_assert(IG_NDIAG * IG_BN <= 512, "the diagonal accumulators must fit the 512 TMEM columns");
static_assert((IG_DIGITS) * IG_KMAX_BLOCKS * (int64_t)IG_KB * 4096 < (int64_t(1) << 31), "s32 diagonal sum overflows");

struct IgDev {
  const int8_t *A, *B;
  const int *ea, *eb;
  int I, J;
  int KB_A, KB_B;   // K blocks per row tile of A / B
  int a_kb, b_kb;   // first K block of this launch within A's / B's range
  int nkb;
  double* out;
  int64_t ldo;
  double alpha;
  int accumulate;
};

__global__ void __launch_bounds__(IG_THREADS, 1) igemm_kernel(const IgDev a) {
  extern __shared__ __align__(1024) unsigned char smem_ig[];
  unsigned char* const smem = smem_ig;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + IG_NSTAGE * IG_STAGE_BYTES);
  uint64_t* s_full = bars;                  // [NSTAGE]
  uint64_t* s_empty = bars + IG_NSTAGE;     // [NSTAGE]
  uint64_t* t_full = bars + 2 * IG_NSTAGE;  // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_full + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tb = blockIdx.x, ta = blockIdx.y;
  if (tid == 0) {
    for (int s = 0; s < IG_NSTAGE; ++s) {
      mma::mbar_init(&s_full[s], 1);
      mma::mbar_init(&s_empty[s], 1);
    }
    mma::mbar_init(t_full, 1);
    mma::fence_barrier_init();
  }
  if (warp == 1) mma::tmem_alloc(tmem_slot, 512);
  mma::tc_fence_before();
  __syncthreads();
  mma::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ======================================================================== producer
    if (lane == 0) {
      const int8_t* pa = a.A + ((size_t)ta * a.KB_A + a.a_kb) * IG_A_BYTES;
      const int8_t* pb = a.B + ((size_t)tb * a.KB_B + a.b_kb) * IG_B_BYTES;
      for (int kb = 0; kb < a.nkb; ++kb) {
        const int s = kb % IG_NSTAGE;
        mma::mbar_wait(&s_empty[s], ((kb / IG_NSTAGE) & 1u) ^ 1u);
        unsigned char* st = smem + (size_t)s * IG_STAGE_BYTES;
        mma::mbar_expect_tx(&s_full[s], IG_STAGE_BYTES);
        mma::bulk_g2s(st, pa + (size_t)kb * IG_A_BYTES, IG_A_BYTES, &s_full[s]);
        mma::bulk_g2s(st + IG_A_BYTES, pb + (size_t)kb * IG_B_BYTES, IG_B_BYTES, &s_full[s]);
      }
    }
  } else if (warp == 1) {
    // ======================================================================== MMA issuer
    // kind::i8: signed int8 A and B (format 1), s32 accumulator (format 2), M = 128; N is set per MMA
    constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(IG_BM >> 4) << 24);
    for (int kb = 0; kb < a.nkb; ++kb) {
      const int s = kb % IG_NSTAGE;
      mma::mbar_wait(&s_full[s], (kb / IG_NSTAGE) & 1u);
      mma::tc_fence_after();
      if (lane == 0) {
        const uint32_t st = mma::smem_u32(smem + (size_t)s * IG_STAGE_BYTES);
#pragma unroll
        for (int da = 0; da < IG_DIGITS; ++da) {
          // A digit da against B digits db = 0 .. 7 - da stacked along N (64 rows each): the products land in
          // the diagonal accumulators da + db, which are adjacent in TMEM - one MMA of N <= 256 per 4 B digits.
          // Piece layout [K half][digit][rows][16 B]: the two K halves lie 8 * rows * 16 B apart (LBO), 8-row
          // core matrices 128 B apart (SBO), across digits too.
          const uint64_t ad = mma::smem_desc(st + da * (IG_BM * 16), IG_DIGITS * IG_BM * 16, 128);
#pragma unroll
          for (int db = 0; db < IG_DIGITS - da; db += 4) {
            const int n = min(4, IG_DIGITS - da - db) * IG_BN;
            const uint64_t bd = mma::smem_desc(st + IG_A_BYTES + db * (IG_BN * 16), IG_DIGITS * IG_BN * 16, 128);
            mma::umma_i8(tmem_base + (uint32_t)((da + db) * IG_BN), ad, bd, IDESC | ((uint32_t)(n >> 3) << 17),
                         (kb > 0 || da > 0) ? 1u : 0u);
          }
        }
        mma::umma_commit(&s_empty[s]);
        if (kb == a.nkb - 1) mma::umma_commit(t_full);
      }
      __syncwarp();
    }
  } else {
    // ======================================================================== epilogue
    const int quarter = warp & 3;   // a warp reads the TMEM lanes 32 (warp % 4) .. + 31
    const int i = ta * IG_BM + quarter * 32 + lane;
    mma::mbar_wait(t_full, 0);
    mma::tc_fence_after();
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int ea = (i < a.I) ? a.ea[i] : 0;
#pragma unroll 1
    for (int cb = 0; cb < IG_BN; cb += 32) {
      double acc[32];
#pragma unroll
      for (int c = 0; c < 32; ++c) acc[c] = 0.0;
#pragma unroll 1
      for (int t = IG_NDIAG - 1; t >= 0; --t) {
        uint32_t v[32];
        mma::tmem_ld32(taddr + (uint32_t)(t * IG_BN + cb), v);
        mma::tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 32; ++c) acc[c] = acc[c] * 0.0078125 + (double)(int)v[c];   // * 2^-7: exact
      }
      if (i < a.I) {
        const int j0 = tb * IG_BN + cb;
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          const int j = j0 + c;
          if (j >= a.J) continue;
          const int eb = a.eb[j];
          const double val = (ea == IG_NONFINITE || eb == IG_NONFINITE) ? CUDART_NAN : a.alpha * ldexp(acc[c], ea + eb);
          double* dst = a.out + (int64_t)i * a.ldo + j;
          *dst = a.accumulate ? *dst + val : val;
        }
      }
    }
  }

  mma::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    mma::tc_fence_after();
    mma::tmem_dealloc(tmem_base, 512);
  }
}

// max |x| of every operand row as the bits of a non-negative double (they order like the values); a NaN counts
// as +Inf.  Not transposed: one block of 256 per row.
__global__ void ig_rowmax_kernel(const double* __restrict__ src, int64_t ld, int kdim,
                                 unsigned long long* __restrict__ mx_bits) {
  __shared__ double sh[256];
  const int row = blockIdx.x;
  double mx = 0.0;
  for (int k = threadIdx.x; k < kdim; k += 256) {
    const double v = fabs(src[(int64_t)row * ld + k]);
    mx = (v == v) ? fmax(mx, v) : CUDART_INF;
  }
  sh[threadIdx.x] = mx;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + w]);
    __syncthreads();
  }
  if (threadIdx.x == 0) mx_bits[row] = (unsigned long long)__double_as_longlong(sh[0]);
}

// transposed (src [kdim, rows]): 32 x 8 threads cover 32 operand rows and one slice of k; slices meet in an
// integer atomicMax
__global__ void ig_rowmax_t_kernel(const double* __restrict__ src, int64_t ld, int rows, int kdim, int kslice,
                                   unsigned long long* __restrict__ mx_bits) {
  __shared__ double sh[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int row = blockIdx.x * 32 + tx;
  const int k0 = blockIdx.y * kslice, k1 = min(kdim, k0 + kslice);
  double mx = 0.0;
  if (row < rows)
    for (int k = k0 + ty; k < k1; k += 8) {
      const double v = fabs(src[(int64_t)k * ld + row]);
      mx = (v == v) ? fmax(mx, v) : CUDART_INF;
    }
  sh[ty][tx] = mx;
  __syncthreads();
  if (ty == 0 && row < rows) {
    for (int y = 1; y < 8; ++y) mx = fmax(mx, sh[y][tx]);
    atomicMax(&mx_bits[row], (unsigned long long)__double_as_longlong(mx));
  }
}

__global__ void ig_rowexp_kernel(const unsigned long long* __restrict__ mx_bits, int rows, int padded,
                                 int* __restrict__ rexp) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= padded) return;
  int e = 0;
  if (row < rows) {
    const double mx = __longlong_as_double((long long)mx_bits[row]);
    if (!isfinite(mx)) {
      e = IG_NONFINITE;
    } else if (mx > 0.0) {
      frexp(mx, &e);
      e -= 6;   // max |x| 2^-e in [32, 64)
    }
  }
  rexp[row] = e;
}

// one thread per (row tile, K block, K half, row): 16 consecutive K positions of one operand row -> 8 digit vectors
template <bool TRANSPOSED>
__global__ void ig_split_kernel(const double* __restrict__ src, int64_t ld, int rows, int kdim, int k0, int kb0, int RT,
                                int KB, int tile, const int* __restrict__ rexp, int8_t* __restrict__ dig) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)RT * KB * 2 * tile) return;
  const int r = (int)(t % tile);
  const int h = (int)((t / tile) & 1);
  const int kb = (int)((t / (2 * tile)) % KB);
  const int rt = (int)(t / (2 * (int64_t)tile * KB));
  const int row = rt * tile + r;
  const int e = rexp[row];
  const int kfirst = (kb0 + kb) * IG_KB + h * 16 - k0;   // src column of the first of the 16 positions
  uint32_t w[IG_DIGITS][4];
#pragma unroll
  for (int da = 0; da < IG_DIGITS; ++da)
#pragma unroll
    for (int q = 0; q < 4; ++q) w[da][q] = 0u;
#pragma unroll
  for (int u = 0; u < 16; ++u) {
    const int k = kfirst + u;
    double y = 0.0;
    if (row < rows && k >= 0 && k < kdim && e != IG_NONFINITE)
      y = ldexp(TRANSPOSED ? src[(int64_t)k * ld + row] : src[(int64_t)row * ld + k], -e);
#pragma unroll
    for (int da = 0; da < IG_DIGITS; ++da) {
      const double d = rint(y);
      w[da][u >> 2] |= ((uint32_t)(int)d & 0xFFu) << (8 * (u & 3));
      y = (y - d) * 128.0;
    }
  }
  int8_t* base = dig + (((size_t)rt * KB + kb) * 2 + h) * IG_DIGITS * tile * 16 + (size_t)r * 16;
#pragma unroll
  for (int da = 0; da < IG_DIGITS; ++da)
    *reinterpret_cast<uint4*>(base + (size_t)da * tile * 16) = make_uint4(w[da][0], w[da][1], w[da][2], w[da][3]);
}

}  // namespace

int dig_from_f64(basq_ctx* ctx, const double* src, int64_t ld, bool transposed, int rows, int kdim, int k0, int tile,
                 DigOperand* op) {
  BASQ_CHECK(rows >= 0 && kdim >= 1 && k0 >= 0 && (tile == IG_BM || tile == IG_BN), BASQ_ERR_INVALID,
             "dig_from_f64: bad shape (rows %d, kdim %d, k0 %d, tile %d)", rows, kdim, k0, tile);
  op->rows = rows;
  op->tile = tile;
  op->RT = std::max(1, ceil_div(rows, tile));
  op->kb0 = k0 / IG_KB;
  op->KB = ceil_div((int64_t)k0 + kdim, IG_KB) - op->kb0;
  const int padded = op->RT * tile;
  BASQ_TRY(op->dig.alloc(ctx, (size_t)op->RT * op->KB * IG_DIGITS * IG_KB * tile));
  BASQ_TRY(op->rexp.alloc(ctx, sizeof(int) * (size_t)padded));
  DevBuf mx;
  BASQ_TRY(mx.alloc(ctx, sizeof(unsigned long long) * (size_t)padded));
  if (rows > 0) {
    if (transposed) {
      BASQ_CUDA(cudaMemsetAsync(mx.p, 0, sizeof(unsigned long long) * (size_t)rows, ctx->stream));
      const int slices = std::max(1, std::min(64, kdim / 128));
      const int kslice = ceil_div(kdim, slices);
      ig_rowmax_t_kernel<<<dim3((unsigned)ceil_div(rows, 32), (unsigned)ceil_div(kdim, kslice)), 256, 0, ctx->stream>>>(
          src, ld, rows, kdim, kslice, mx.as<unsigned long long>());
    } else {
      ig_rowmax_kernel<<<rows, 256, 0, ctx->stream>>>(src, ld, kdim, mx.as<unsigned long long>());
    }
    ctx->launches++;
  }
  ig_rowexp_kernel<<<ceil_div(padded, 256), 256, 0, ctx->stream>>>(mx.as<unsigned long long>(), rows, padded,
                                                                   op->rexp.as<int>());
  const int64_t total = (int64_t)op->RT * op->KB * 2 * tile;
  const unsigned grid = (unsigned)ceil_div64(total, 256);
  if (transposed)
    ig_split_kernel<true><<<grid, 256, 0, ctx->stream>>>(src, ld, rows, kdim, k0, op->kb0, op->RT, op->KB, tile,
                                                         op->rexp.as<int>(), op->dig.as<int8_t>());
  else
    ig_split_kernel<false><<<grid, 256, 0, ctx->stream>>>(src, ld, rows, kdim, k0, op->kb0, op->RT, op->KB, tile,
                                                          op->rexp.as<int>(), op->dig.as<int8_t>());
  ctx->launches += 2;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;   // `mx` returns to the context's block cache; stream order keeps it intact until it has been read
}

int igemm(basq_ctx* ctx, const DigOperand& A, const DigOperand& B, double alpha, double* out, int64_t ldo,
          bool accumulate) {
  BASQ_CHECK(A.tile == IG_BM && B.tile == IG_BN, BASQ_ERR_INVALID, "igemm: operand tiles %d / %d (need %d / %d)", A.tile,
             B.tile, IG_BM, IG_BN);
  BASQ_CHECK(B.kb0 >= A.kb0 && B.kb0 + B.KB <= A.kb0 + A.KB, BASQ_ERR_INVALID,
             "igemm: K blocks [%d, %d) of B lie outside A's [%d, %d)", B.kb0, B.kb0 + B.KB, A.kb0, A.kb0 + A.KB);
  BASQ_CHECK((size_t)IG_SMEM <= ctx->smem_optin, BASQ_ERR_UNSUPPORTED, "igemm: needs %d B shared memory", IG_SMEM);
  if (A.rows <= 0 || B.rows <= 0) return BASQ_OK;
  IgDev d;
  d.A = A.dig.as<int8_t>(); d.B = B.dig.as<int8_t>();
  d.ea = A.rexp.as<int>(); d.eb = B.rexp.as<int>();
  d.I = A.rows; d.J = B.rows;
  d.KB_A = A.KB; d.KB_B = B.KB;
  d.out = out; d.ldo = ldo;
  d.alpha = alpha;
  BASQ_CUDA(cudaFuncSetAttribute(igemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, IG_SMEM));
  // one launch per K range whose diagonal sums stay exact in s32; the ranges add in fp64
  for (int kb = 0; kb < B.KB; kb += IG_KMAX_BLOCKS) {
    d.b_kb = kb;
    d.a_kb = B.kb0 - A.kb0 + kb;
    d.nkb = std::min(IG_KMAX_BLOCKS, B.KB - kb);
    d.accumulate = (accumulate || kb > 0) ? 1 : 0;
    igemm_kernel<<<dim3((unsigned)B.RT, (unsigned)A.RT), IG_THREADS, IG_SMEM, ctx->stream>>>(d);
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
  }
  return BASQ_OK;
}

}  // namespace basq
