// Weighted set sums of Gram columns on the 5th-generation tensor cores (fp32 data, linear modes).
//
//   G[m, j] (+)= sum over local points p with (off + p) mod S == j of  w_p * k(z_m, x_p)
//
// The exponent argument of every kernel family is bilinear in prepared operands,
//   arg(m, p) = a_p + b_m + sum_i x'_{p,i} zz_{m,i}        (see common.cuh: KParams),
// so a 128-landmark x NT-point tile of arguments is ONE small GEMM with K = 3 DP + 6 (padded to the MMA's K step):
//   * x' and zz are split into fp16 "hi + lo" parts with 11 significant bits each (kind::f16: K = 48 at
//     d = 10, three MMAs per tile), and the three significant cross products (hi hi, lo hi, hi lo) occupy
//     three K columns per dimension (~2^-21 relative).  fp16's range is enough for centred,
//     lengthscale-scaled coordinates (values beyond +-6e4 are clamped: such pairs have k = 0 either way);
//     pieces below 6e-5 lose bits to the subnormal spacing 6e-8, an absolute 3e-8 |zz| per term of the
//     argument - below its fp32 rounding;
//   * a_p and b_m ride along as three pieces each against constant-one columns.
// tcgen05.mma (M = 128, N = NT, operands K-major in shared memory, no swizzle) writes the
// argument tile into TMEM; the epilogue warps read it back with tcgen05.ld, apply exp2 / the Matern
// polynomial on the MUFU/FMA pipes and accumulate w_p * k in fp64 - one accumulator per (landmark,
// set).  What remains on the CUDA cores per pair is 1 MUFU + 2 integer ops + 1 DFMA; the DP-long
// FFMA chain of the scalar kernel moved to the tensor pipe.
//
// CTA = 20 warps, one CTA per SM, persistent over work items (MT landmark tiles x JT sets).  (20, not
// 21: registers are allotted per group of 4 warps, so a 21st warp would cap every thread at 80
// registers instead of 96 - measured 42.2 -> 39.3 ms for the round-1 sweep.)
//   warps 0-15  epilogue: warp w owns TMEM lanes 32 (w % 4) .. +31 (read as 16x256b fragments: four
//               landmarks x two sets per thread) and column part w / 4 of every accumulator buffer
//               (4 warps per scheduler hide the tcgen05.ld / MUFU / DFMA latencies of one another;
//               the MUFU pipe is the bound)
//   warps 16-18 producers: candidate records (HBM/L2) -> hi/lo split -> K-major B stage in smem
//   warp  19    TMEM allocation, landmark (A) tile bulk copies, tcgen05.mma issue (one lane)
// Pipelines (mbarriers): B stages full/empty (3-deep ring), TMEM accumulators full/empty (2 buffers),
// A tiles full/empty.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace basq {

struct SetSumMmaDev {
  const unsigned char* recs;
  int64_t count;
  int64_t off;
  int S;
  int64_t p_lo, p_hi;
  const float* lmA;  // [n_mtiles_alloc][KA/8][128][8 halves] landmark operand, tile-blocked
  int Mtot;
  int n_mgroups;     // ceil(Mtot / (MT * 128))
  int n_jgroups;     // ceil(S / JT)
  float os_f;
  double* G;
  int64_t ldg;
  int accumulate;
  double grid_m;     // reproducible instances: 1.5 * 2^52 * Q of the pass's grid Q (grid_round, common.cuh)
};

template <int DP>
struct MmaCfg {
  static constexpr int KA = (3 * DP + 6 + 15) / 16 * 16;  // K columns (multiple of the MMA K, 16)
  static constexpr int NT = KA <= 80 ? 256 : 128;      // points per tile (MMA N)
  static constexpr int MT = KA > 160 ? 1 : 2;          // landmark tiles (of 128) per work item
  static constexpr int JT = 8;                         // sets per work item
  static constexpr int EC = NT / JT;                   // set members per tile
  static constexpr int NSTAGE = 3;
  static constexpr int RB = ((24 + 4 * DP) + 15) / 16 * 16;  // record bytes (rec_bytes_f32)
  static constexpr int A_TILE_BYTES = KA * 128 * 2;   // fp16 operands
  static constexpr int B_STAGE_BYTES = KA * NT * 2;
  static constexpr int W_STAGE_BYTES = NT * 8;
#ifndef BASQ_EPI_WARPS
#define BASQ_EPI_WARPS 16
#endif
  static constexpr int EPI_WARPS = BASQ_EPI_WARPS, PROD_WARPS = 3;  // 20 warps: registers are allotted per 4 warps, 21 would cap a thread at 80
  static constexpr int NPART = EPI_WARPS / 4;          // column parts of an accumulator buffer (one warp each per lane quarter)
  static constexpr int COMB_SLOT_BYTES = MT * 128 * JT * 8;
  static constexpr int SMEM_FIXED = MT * A_TILE_BYTES + NSTAGE * (B_STAGE_BYTES + W_STAGE_BYTES) + 256;
  // End-of-item combine of the column parts.  With one slot per part (NPART - 1 slots) the parts
  // hand their partial sums over with ONE arrive and go on to the next item while part 0 sums and
  // writes G; with a single slot (large DP: no room) they take turns under full barriers.
  static constexpr int NSLOT = (SMEM_FIXED + (NPART - 1) * COMB_SLOT_BYTES <= 227 * 1024) ? NPART - 1 : 1;
  static constexpr int COMB_BYTES = NSLOT * COMB_SLOT_BYTES;
  // landmark tiles are double-buffered (the next work item's tiles arrive while this item's MMAs
  // run) whenever a second copy still fits the 227 KB of shared memory
  static constexpr int NABUF = (SMEM_FIXED + COMB_BYTES + MT * A_TILE_BYTES <= 227 * 1024) ? 2 : 1;
  static constexpr int OFF_A = 0;
  static constexpr int OFF_B = OFF_A + NABUF * MT * A_TILE_BYTES;
  static constexpr int OFF_W = OFF_B + NSTAGE * B_STAGE_BYTES;
  static constexpr int OFF_COMB = OFF_W + NSTAGE * W_STAGE_BYTES;
  static constexpr int OFF_BAR = OFF_COMB + COMB_BYTES;
  static constexpr int SMEM_BYTES = OFF_BAR + 256;
  static constexpr int TMEM_COLS = 2 * NT;             // two accumulator buffers (256 or 512)
  static constexpr int THREADS = (EPI_WARPS + PROD_WARPS + 1) * 32;
};

namespace mma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(b)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, fp16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, signed int8 inputs, exact s32 accumulate
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// K-major operand without swizzle, stored as [K / 8][rows][8 halves]: 8-row core matrices are
// contiguous (SBO = 128 B), the next 16-byte K chunk lies one plane further (LBO = rows * 16 B).
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  return d;
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// 16 lanes x 32 columns: thread T receives rows T/4 and T/4 + 8 of the 16 lanes at the address and, of
// every group of 8 columns k, columns 2 (T%4) and 2 (T%4) + 1 (v[4k+0..1] row T/4, v[4k+2..3] row T/4 + 8)
__device__ __forceinline__ void tmem_ld16x256_x4(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// fp16 pieces of an fp32 value: hi = the value cut to 11 significant bits (exact in fp16 within its normal
// range), lo = the remainder rounded to fp16 (sum reproduces the value to ~2^-22); values are clamped to
// fp16's range first
__device__ __forceinline__ float clamp_h(float v) { return fminf(fmaxf(v, -60000.f), 60000.f); }
__device__ __forceinline__ void split2h(float v, __half& hi, __half& lo) {
  v = clamp_h(v);
  const float t = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
  hi = __float2half_rn(t);
  lo = __float2half_rn(__fsub_rn(v, __half2float(hi)));
}
__device__ __forceinline__ void split3h(float v, __half& p1, __half& p2, __half& p3) {
  v = clamp_h(v);
  p1 = __float2half_rn(v);
  const float r = __fsub_rn(v, __half2float(p1));
  p2 = __float2half_rn(r);
  p3 = __float2half_rn(__fsub_rn(r, __half2float(p2)));
}

}  // namespace mma

// ---------------------------------------------------------------------------------------------
// landmark operand: lmA[tile][kc][row][8 halves] from the prepared zz [Mtot, DP] / b [Mtot]
//   K column 3i   : zz_hi_i   (x hi)      3i+1 : zz_hi_i  (x lo)      3i+2 : zz_lo_i  (x hi)
//   3DP .. 3DP+2  : 1 (a pieces)          3DP+3 .. 3DP+5 : b pieces (x 1)      rest : 0
// ---------------------------------------------------------------------------------------------
template <int DP>
__global__ void build_lmA_kernel(const float* __restrict__ zz, const float* __restrict__ bz, int Mtot, int n_tiles,
                                 float* __restrict__ lmA) {
  using Cfg = MmaCfg<DP>;
  constexpr int KA = Cfg::KA;
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n_tiles * 128) return;
  const int tile = m >> 7, row = m & 127;
  __half vals[KA];
#pragma unroll
  for (int k = 0; k < KA; ++k) vals[k] = __float2half_rn(0.f);
  if (m < Mtot) {
#pragma unroll
    for (int i = 0; i < DP; ++i) {
      __half zh, zl;
      mma::split2h(zz[(int64_t)m * DP + i], zh, zl);
      vals[3 * i] = zh;
      vals[3 * i + 1] = zh;
      vals[3 * i + 2] = zl;
    }
    vals[3 * DP] = vals[3 * DP + 1] = vals[3 * DP + 2] = __float2half_rn(1.f);
    mma::split3h(bz[m], vals[3 * DP + 3], vals[3 * DP + 4], vals[3 * DP + 5]);
  }
  uint4* dst = reinterpret_cast<uint4*>(lmA) + (int64_t)tile * (KA / 8) * 128 + row;
#pragma unroll
  for (int kc = 0; kc < KA / 8; ++kc) dst[kc * 128] = *reinterpret_cast<const uint4*>(&vals[8 * kc]);
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
// REPRO: every term w_p k is rounded to the pass's grid before it is added, so that the sums are exact and do
// not depend on the tiling or on how the points are split over ranks (DESIGN.md, reproducible mode)
template <int FAM, int DP, bool REPRO>
__global__ void __launch_bounds__(MmaCfg<DP>::THREADS, 1) setsum_mma_kernel(const SetSumMmaDev a) {
  using Cfg = MmaCfg<DP>;
  constexpr int KA = Cfg::KA, NT = Cfg::NT, MT = Cfg::MT, JT = Cfg::JT, EC = Cfg::EC, NSTAGE = Cfg::NSTAGE,
                RB = Cfg::RB;
  extern __shared__ __align__(1024) unsigned char smem_mma[];
  unsigned char* const smem = smem_mma;
  unsigned char* sA = smem + Cfg::OFF_A;
  unsigned char* sB = smem + Cfg::OFF_B;
  double* sW = reinterpret_cast<double*>(smem + Cfg::OFF_W);
  double* sComb = reinterpret_cast<double*>(smem + Cfg::OFF_COMB);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* b_full = bars;               // [NSTAGE]
  uint64_t* b_empty = bars + NSTAGE;     // [NSTAGE]
  uint64_t* t_full = bars + 2 * NSTAGE;  // [2]
  uint64_t* t_empty = t_full + 2;        // [2]
  uint64_t* a_full = t_empty + 2;        // [2]
  uint64_t* a_empty = a_full + 2;        // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_empty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) {
      mma::mbar_init(&b_full[s], Cfg::PROD_WARPS * 32);
      mma::mbar_init(&b_empty[s], 1 + Cfg::EPI_WARPS);
    }
    for (int b = 0; b < 2; ++b) {
      mma::mbar_init(&t_full[b], 1);
      mma::mbar_init(&t_empty[b], Cfg::EPI_WARPS);
    }
    for (int b = 0; b < 2; ++b) {
      mma::mbar_init(&a_full[b], 1);
      mma::mbar_init(&a_empty[b], 1);
    }
    mma::fence_barrier_init();
  }
  if (warp == Cfg::EPI_WARPS + Cfg::PROD_WARPS) mma::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  mma::tc_fence_before();
  __syncthreads();
  mma::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int64_t S = a.S;
  const int n_items = a.n_mgroups * a.n_jgroups;

  // member range [e_lo, e_hi) of the JT sets starting at j0 that falls into [p_lo, p_hi)
  auto item_range = [&](int j0, int64_t& e_lo, int64_t& n_tiles) {
    const int64_t num_lo = a.p_lo + a.off - (int64_t)(j0 + JT - 1);
    e_lo = num_lo <= 0 ? 0 : (num_lo + S - 1) / S;
    const int64_t num_hi = a.p_hi - 1 + a.off - (int64_t)j0;
    const int64_t e_hi = num_hi < 0 ? 0 : num_hi / S + 1;
    const int64_t n_e = e_hi > e_lo ? e_hi - e_lo : 0;
    n_tiles = (n_e + EC - 1) / EC;
  };

  if (warp < Cfg::EPI_WARPS) {
    // ======================================================================== epilogue
    // Accumulator fragments are read with the 16x256b shape: a thread then owns 4 landmarks (rows
    // r0 + {0, 8, 16, 24}) and, with JT = 8 sets interleaved over the columns, exactly TWO sets
    // (2 (lane % 4) and the next one) - so one 16-byte weight load serves 8 evaluations, and the
    // thread still carries MT * 4 * 2 = MT * JT accumulators.
    static_assert(JT == 8, "the fragment mapping below assumes 8 sets per work item");
    const int quarter = warp & 3, part = warp >> 2;
    const int r0 = quarter * 32 + (lane >> 2);   // first of the thread's four rows (within the 128-row tile)
    const int s0 = 2 * (lane & 3);               // first of the thread's two sets
    constexpr int NPART = Cfg::NPART;
    constexpr int PART_COLS = NT / NPART;
    static_assert(PART_COLS % 32 == 0, "column part must be a multiple of the tcgen05.ld width");
    uint32_t it = 0, tc = 0, items_done = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int mg = item % a.n_mgroups, jg = item / a.n_mgroups;
      const int j0 = jg * JT;
      int64_t e_lo, n_tiles;
      item_range(j0, e_lo, n_tiles);
      double acc[MT][4][2];  // [landmark tile][row slot: r0 + 8 * slot][set s0 + {0, 1}]
#pragma unroll
      for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int rs = 0; rs < 4; ++rs) acc[mt][rs][0] = acc[mt][rs][1] = 0.0;
      for (int64_t t = 0; t < n_tiles; ++t, ++it) {
        const int stage = it % NSTAGE;
        const double* wst = sW + stage * NT + part * PART_COLS + s0;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt, ++tc) {
          const uint32_t buf = tc & 1u;
          mma::mbar_wait(&t_full[buf], (tc >> 1) & 1u);
          mma::tc_fence_after();
          const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * NT + part * PART_COLS;
#pragma unroll
          for (int cb = 0; cb < PART_COLS; cb += 32) {
            uint32_t va[16], vb[16];
            mma::tmem_ld16x256_x4(taddr + cb, va);                         // lanes +0 .. +15
            mma::tmem_ld16x256_x4(taddr + ((uint32_t)16 << 16) + cb, vb);  // lanes +16 .. +31
            mma::tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const double2 w2 = *reinterpret_cast<const double2*>(wst + cb + 8 * k);
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                // row slots 2 h and 2 h + 1
                const float u00 = __uint_as_float(h ? vb[4 * k + 0] : va[4 * k + 0]);
                const float u01 = __uint_as_float(h ? vb[4 * k + 1] : va[4 * k + 1]);
                const float u10 = __uint_as_float(h ? vb[4 * k + 2] : va[4 * k + 2]);
                const float u11 = __uint_as_float(h ? vb[4 * k + 3] : va[4 * k + 3]);
                const float k00 = finish_f32(FAM, u00, a.os_f), k01 = finish_f32(FAM, u01, a.os_f);
                const float k10 = finish_f32(FAM, u10, a.os_f), k11 = finish_f32(FAM, u11, a.os_f);
                if (REPRO) {
                  acc[mt][2 * h][0] += grid_round(f2d_pos(k00), w2.x, a.grid_m);
                  acc[mt][2 * h][1] += grid_round(f2d_pos(k01), w2.y, a.grid_m);
                  acc[mt][2 * h + 1][0] += grid_round(f2d_pos(k10), w2.x, a.grid_m);
                  acc[mt][2 * h + 1][1] += grid_round(f2d_pos(k11), w2.y, a.grid_m);
                } else {
                  acc[mt][2 * h][0] = fma(f2d_pos(k00), w2.x, acc[mt][2 * h][0]);
                  acc[mt][2 * h][1] = fma(f2d_pos(k01), w2.y, acc[mt][2 * h][1]);
                  acc[mt][2 * h + 1][0] = fma(f2d_pos(k10), w2.x, acc[mt][2 * h + 1][0]);
                  acc[mt][2 * h + 1][1] = fma(f2d_pos(k11), w2.y, acc[mt][2 * h + 1][1]);
                }
              }
            }
          }
          mma::tc_fence_before();
          __syncwarp();
          if (lane == 0) mma::mbar_arrive(&t_empty[buf]);
        }
        // the weights of this stage have been consumed by this warp
        __syncwarp();
        if (lane == 0) mma::mbar_arrive(&b_empty[stage]);
      }
      // ---- combine the column parts in a fixed order (deterministic sums) and write G
      // the thread's accumulator (mt, rs, c) belongs to tile row r0 + 8 rs and set s0 + c
      constexpr int SLOT = MT * 128 * JT;
      constexpr bool HANDOVER = (Cfg::NSLOT == NPART - 1);
      auto slot_of = [&](int mt, int rs, int c) { return (mt * JT + s0 + c) * 128 + r0 + 8 * rs; };
      if (HANDOVER) {
        if (part > 0) {
          if (items_done > 0) mma::named_bar_sync(2, Cfg::EPI_WARPS * 32);  // part 0 is done with the previous sums
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int rs = 0; rs < 4; ++rs)
#pragma unroll
              for (int c = 0; c < 2; ++c) sComb[(part - 1) * SLOT + slot_of(mt, rs, c)] = acc[mt][rs][c];
          __threadfence_block();
          mma::named_bar_arrive(1, Cfg::EPI_WARPS * 32);
        } else {
          mma::named_bar_sync(1, Cfg::EPI_WARPS * 32);
        }
      } else {
#pragma unroll
        for (int pp = NPART - 1; pp >= 1; --pp) {
          if (part == pp) {
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
              for (int rs = 0; rs < 4; ++rs)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                  double* d = &sComb[slot_of(mt, rs, c)];
                  *d = (pp == NPART - 1) ? acc[mt][rs][c] : (*d + acc[mt][rs][c]);
                }
          }
          mma::named_bar_sync(1, Cfg::EPI_WARPS * 32);
        }
      }
      if (part == 0) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int rs = 0; rs < 4; ++rs) {
            const int m = (mg * MT + mt) * 128 + r0 + 8 * rs;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              double others;
              if (HANDOVER) {
                others = sComb[(NPART - 2) * SLOT + slot_of(mt, rs, c)];
#pragma unroll
                for (int pp = NPART - 3; pp >= 0; --pp) others += sComb[pp * SLOT + slot_of(mt, rs, c)];
              } else {
                others = sComb[slot_of(mt, rs, c)];
              }
              const int j = j0 + s0 + c;
              if (m < a.Mtot && j < a.S) {
                const double v = acc[mt][rs][c] + others;
                double* dst = a.G + (int64_t)m * a.ldg + j;
                *dst = a.accumulate ? (*dst + v) : v;
              }
            }
          }
        if (HANDOVER) mma::named_bar_arrive(2, Cfg::EPI_WARPS * 32);
      }
      if (!HANDOVER) mma::named_bar_sync(1, Cfg::EPI_WARPS * 32);
      ++items_done;
    }
  } else if (warp < Cfg::EPI_WARPS + Cfg::PROD_WARPS) {
    // ======================================================================== producers
    const int ptid = tid - Cfg::EPI_WARPS * 32;
    constexpr int NPROD = Cfg::PROD_WARPS * 32;
    uint32_t it = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int jg = item / a.n_mgroups;
      const int j0 = jg * JT;
      int64_t e_lo, n_tiles;
      item_range(j0, e_lo, n_tiles);
      for (int64_t t = 0; t < n_tiles; ++t, ++it) {
        const int stage = it % NSTAGE;
        mma::mbar_wait(&b_empty[stage], ((it / NSTAGE) & 1u) ^ 1u);
        uint4* bst = reinterpret_cast<uint4*>(sB + (size_t)stage * Cfg::B_STAGE_BYTES);
        double* wst = sW + stage * NT;
#pragma unroll
        for (int c = ptid; c < NT; c += NPROD) {
          const int ei = c / JT, jj = c % JT;
          const int64_t e = e_lo + t * EC + ei;
          const int64_t p = (int64_t)(j0 + jj) + e * S - a.off;
          const bool ok = (j0 + jj < a.S) && (p >= a.p_lo) && (p < a.p_hi);
          double w = 0.0;
          constexpr int NV = RB / 16;
          uint4 q[NV];
#pragma unroll
          for (int v = 0; v < NV; ++v) q[v] = make_uint4(0u, 0u, 0u, 0u);
          if (ok) {
            const uint4* rec = reinterpret_cast<const uint4*>(a.recs + p * RB);
#pragma unroll
            for (int v = 0; v < NV; ++v) q[v] = __ldg(rec + v);
            w = __hiloint2double((int)q[0].y, (int)q[0].x);
          }
          float f[(NV - 1) * 4];  // [idx, a, x0, x1, ...]
#pragma unroll
          for (int v = 1; v < NV; ++v) {
            f[(v - 1) * 4 + 0] = __uint_as_float(q[v].x);
            f[(v - 1) * 4 + 1] = __uint_as_float(q[v].y);
            f[(v - 1) * 4 + 2] = __uint_as_float(q[v].z);
            f[(v - 1) * 4 + 3] = __uint_as_float(q[v].w);
          }
          // pieces as floats first (hi = the value cut to 11 significant bits by a mask, lo = the exact fp32
          // remainder), then packed pair conversions only: scalar float <-> half conversions run on the
          // 16-lane pipe of the epilogue's ex2 - the pipe that bounds this kernel
          float fv[KA];
#pragma unroll
          for (int k = 0; k < KA; ++k) fv[k] = 0.f;
          if (ok) {
#pragma unroll
            for (int i = 0; i < DP; ++i) {
              const float x = mma::clamp_h(f[2 + i]);
              const float xh = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
              fv[3 * i] = xh;
              fv[3 * i + 1] = __fsub_rn(x, xh);
              fv[3 * i + 2] = xh;
            }
            const float av = mma::clamp_h(f[1]);
            const float a1 = __uint_as_float(__float_as_uint(av) & 0xFFFFE000u);
            const float r1 = __fsub_rn(av, a1);
            const float a2 = __uint_as_float(__float_as_uint(r1) & 0xFFFFE000u);
            fv[3 * DP] = a1;
            fv[3 * DP + 1] = a2;
            fv[3 * DP + 2] = __fsub_rn(r1, a2);
            fv[3 * DP + 3] = fv[3 * DP + 4] = fv[3 * DP + 5] = 1.f;
          }
#pragma unroll
          for (int kc = 0; kc < KA / 8; ++kc) {
            __half2 h2[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) h2[u] = __floats2half2_rn(fv[8 * kc + 2 * u], fv[8 * kc + 2 * u + 1]);
            bst[kc * NT + c] = *reinterpret_cast<const uint4*>(h2);
          }
          wst[c] = w;
        }
        mma::fence_proxy_async();
        mma::mbar_arrive(&b_full[stage]);
      }
    }
  } else {
    // ======================================================================== MMA issuer
    // instruction descriptor: D fp32 (bit 4), A / B fp16 (formats 0), K-major both; N, M
    constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(NT >> 3) << 17) | ((128u >> 4) << 24);
    constexpr int NABUF = Cfg::NABUF;
    uint32_t it = 0, tc = 0, ac = 0;  // ac counts the work items with tiles (= landmark tile loads)
    auto next_item = [&](int item) {  // first item >= `item` of this CTA that has tiles; n_items if none
      for (; item < n_items; item += gridDim.x) {
        int64_t e_lo, n_tiles;
        item_range((item / a.n_mgroups) * JT, e_lo, n_tiles);
        if (n_tiles > 0) break;
      }
      return item < n_items ? item : n_items;
    };
    // request the landmark tiles of work item `item` as load number `ld` (buffer ld % NABUF)
    auto load_A = [&](int item, uint32_t ld) {
      const uint32_t ab = ld % NABUF, use = ld / NABUF;
      if (use > 0) mma::mbar_wait(&a_empty[ab], (use - 1) & 1u);  // the buffer's previous item has issued all MMAs
      if (lane == 0) {
        const int mg = item % a.n_mgroups;
        mma::mbar_expect_tx(&a_full[ab], MT * Cfg::A_TILE_BYTES);
        mma::bulk_g2s(sA + ab * MT * Cfg::A_TILE_BYTES, a.lmA + (size_t)mg * MT * (Cfg::A_TILE_BYTES / 4),
                      MT * Cfg::A_TILE_BYTES, &a_full[ab]);
      }
    };
    int item = next_item(blockIdx.x);
    if (item < n_items) load_A(item, 0);
    while (item < n_items) {
      const int jg = item / a.n_mgroups;
      int64_t e_lo, n_tiles;
      item_range(jg * JT, e_lo, n_tiles);
      const int nxt = next_item(item + gridDim.x);
      if (NABUF == 2 && nxt < n_items) load_A(nxt, ac + 1);
      const uint32_t ab = ac % NABUF;
      mma::mbar_wait(&a_full[ab], (ac / NABUF) & 1u);
      unsigned char* const sAcur = sA + ab * MT * Cfg::A_TILE_BYTES;
      for (int64_t t = 0; t < n_tiles; ++t, ++it) {
        const int stage = it % NSTAGE;
        mma::mbar_wait(&b_full[stage], (it / NSTAGE) & 1u);
        mma::tc_fence_after();
#pragma unroll
        for (int mt = 0; mt < MT; ++mt, ++tc) {
          const uint32_t buf = tc & 1u;
          mma::mbar_wait(&t_empty[buf], ((tc >> 1) & 1u) ^ 1u);
          mma::tc_fence_after();
          if (lane == 0) {
            const uint32_t a_base = mma::smem_u32(sAcur + mt * Cfg::A_TILE_BYTES);
            const uint32_t b_base = mma::smem_u32(sB + (size_t)stage * Cfg::B_STAGE_BYTES);
#pragma unroll
            for (int ks = 0; ks < KA / 16; ++ks) {   // one MMA (K = 16) = two 16-byte K chunks
              const uint64_t ad = mma::smem_desc(a_base + ks * 2 * (128 * 16), 128 * 16, 128);
              const uint64_t bd = mma::smem_desc(b_base + ks * 2 * (NT * 16), NT * 16, 128);
              mma::umma_f16(tmem_base + buf * NT, ad, bd, IDESC, ks > 0 ? 1u : 0u);
            }
            mma::umma_commit(&t_full[buf]);
          }
          __syncwarp();
        }
        if (lane == 0) mma::umma_commit(&b_empty[stage]);
        __syncwarp();
      }
      if (lane == 0) mma::umma_commit(&a_empty[ab]);
      __syncwarp();
      ++ac;
      if (NABUF == 1 && nxt < n_items) load_A(nxt, ac);
      item = nxt;
    }
  }

  mma::tc_fence_before();
  __syncthreads();
  if (warp == Cfg::EPI_WARPS + Cfg::PROD_WARPS) {
    mma::tc_fence_after();
    mma::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int FAM, int DP, bool REPRO>
int launch_setsum_mma_inst(basq_ctx* ctx, SetSumMmaDev dev) {
  using Cfg = MmaCfg<DP>;
  dev.n_mgroups = ceil_div(dev.Mtot, Cfg::MT * 128);
  dev.n_jgroups = ceil_div(dev.S, Cfg::JT);
  const int64_t n_items = (int64_t)dev.n_mgroups * dev.n_jgroups;
  BASQ_CHECK(n_items < (1ll << 31), BASQ_ERR_UNSUPPORTED, "set_sums: too many work items");
  BASQ_CHECK((size_t)Cfg::SMEM_BYTES <= ctx->smem_optin, BASQ_ERR_UNSUPPORTED,
             "set_sums: kernel needs %d B shared memory (limit %zu)", Cfg::SMEM_BYTES, ctx->smem_optin);
  BASQ_CUDA(cudaFuncSetAttribute(setsum_mma_kernel<FAM, DP, REPRO>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 Cfg::SMEM_BYTES));
  const int grid = (int)std::min<int64_t>(ctx->num_sms, n_items);
  setsum_mma_kernel<FAM, DP, REPRO><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, ctx->stream>>>(dev);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

template <int FAM, int DP>
int launch_setsum_mma_dp(basq_ctx* ctx, const SetSumMmaDev& dev) {
  return dev.grid_m != 0.0 ? launch_setsum_mma_inst<FAM, DP, true>(ctx, dev) : launch_setsum_mma_inst<FAM, DP, false>(ctx, dev);
}

template <int FAM>
int launch_setsum_mma_family(basq_ctx* ctx, int dp, const SetSumMmaDev& dev) {
  switch (dp) {
    case 2: return launch_setsum_mma_dp<FAM, 2>(ctx, dev);
    case 4: return launch_setsum_mma_dp<FAM, 4>(ctx, dev);
    case 6: return launch_setsum_mma_dp<FAM, 6>(ctx, dev);
    case 8: return launch_setsum_mma_dp<FAM, 8>(ctx, dev);
    case 10: return launch_setsum_mma_dp<FAM, 10>(ctx, dev);
    case 12: return launch_setsum_mma_dp<FAM, 12>(ctx, dev);
    case 16: return launch_setsum_mma_dp<FAM, 16>(ctx, dev);
    case 20: return launch_setsum_mma_dp<FAM, 20>(ctx, dev);
    case 24: return launch_setsum_mma_dp<FAM, 24>(ctx, dev);
    case 32: return launch_setsum_mma_dp<FAM, 32>(ctx, dev);
  }
  set_error("set_sums: no tensor-core kernel compiled for padded dimension %d", dp);
  return BASQ_ERR_UNSUPPORTED;
}

template <int DP>
int launch_build_lmA_dp(basq_ctx* ctx, const float* zz, const float* bz, int Mtot, int n_tiles, float* lmA) {
  build_lmA_kernel<DP><<<ceil_div((int64_t)n_tiles * 128, 128), 128, 0, ctx->stream>>>(zz, bz, Mtot, n_tiles, lmA);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

// one definition per translation unit (setsum_mma_*.cu)
int launch_setsum_mma_rbf(basq_ctx*, int, const SetSumMmaDev&);
int launch_setsum_mma_m15(basq_ctx*, int, const SetSumMmaDev&);
int launch_setsum_mma_m25(basq_ctx*, int, const SetSumMmaDev&);
// allocation size (floats) and tile count of the landmark operand for `count` landmarks
int lmA_tiles(int dp, int count);
size_t lmA_floats(int dp, int count);
int build_lmA(basq_ctx* ctx, int dp, const float* zz, const float* bz, int Mtot, float* lmA);

}  // namespace basq
