// Weighted set sums for the pairwise NON-LINEAR kernels (WSABI-M, MMLT) on the tensor cores.
//
//   G[m, j] = sum over local points p of cell j of  mu_p * nl( C(z_m, x_p) ),
//   C(z, x) = k(z, x) - sum_o Az[m, o] k(xobs_o, x),      Az = K(Z, Xobs) W          (BASQ/_gp.py:259-277)
//   nl(C)   = m(z) m(x) C + C^2 / 2   (wsabim_kernel, BASQ/_wsabi.py:228-249)
//           = mu_g(z) mu_g(x) (exp(C) - 1)   (gspace_kernel, SOBER/BASQ/_scale_mmlt.py:258-278)
//
// The non-linearity needs C per (landmark, candidate) pair, so the posterior correction cannot be
// folded into the projection as in the linear modes: it is a GEMM of Az [M x n_obs] against
// k(Xobs, X) [n_obs x N] - 2 n_obs flop per pair, 2e14 flop for one sweep of config 5 - and the one
// place on this path where the tensor pipe is the bound.  Two kernels per chunk of cells:
//
//   kxgen_kernel   k(Xobs, x_p) for the chunk's candidates on the CUDA cores (n_obs evaluations per
//                  candidate, ~1 % of the work), written as the B operand of the GEMM: fp16 "hi + lo"
//                  split (hi = fp16(v), lo = fp16(v - hi), v = k 2^sB in [0, 2^14]), tile-blocked
//                  K-major [tile of 256 candidates][K / 8][256][8 halves] so that one (tile, 32-wide K
//                  block) is a contiguous 16 KB piece for cp.async.bulk.  The tile's candidate records
//                  are copied next to it (invalid slots get weight 0).  A chunk is sized to stay
//                  L2-resident while the 79 landmark tiles of M = 1e4 re-read it.
//   nlsum_kernel   persistent, one CTA per SM, 11 warps:
//                    warp 8   streams 48 KB stages (Az hi / lo 8 KB each, kx hi / lo 16 KB each) of one
//                             32-wide K block with cp.async.bulk into a 3-deep ring
//                    warp 9   one lane issues tcgen05.mma kind::f16 (M = 128 landmarks, N = 256
//                             candidates, K = 16): three products per K step (lo hi, hi lo, hi hi: the fp32
//                             product to ~2^-21, fp32 accumulation in TMEM), 2 x 256 TMEM columns so that
//                             the epilogue of one tile overlaps the MMAs of the next
//                    warp 10  streams the tile's candidate records (16 KB) into shared memory
//                    warps 0-7 epilogue: tcgen05.ld the correction, k(z_m, x_p) on the FMA / MUFU pipes
//                             with the library's one operation sequence (pair_eval_f32), C, the
//                             non-linearity in fp32, exact widening, fp64 accumulation per (landmark,
//                             set); column halves are combined in a fixed order and written to G.
//                  SETSUM mode interleaves 8 sets x 32 members over a tile's columns (as the linear
//                  kernel does); GRAM mode (cells with at most one member: features, final stage)
//                  gives every column its own cell and writes mu_p nl(C) straight to G.
//
// Accuracy: Az rows are scaled by a power of two to [2^13, 2^14) and split in fp64; kx is split from
// its fp32 value; the dropped lo lo product and the fp32 accumulator leave ~2^-21 |Az_m|_1 relative to
// the outputscale - the same amplification the fp32 kernel values themselves carry (eps_k |Az_m|_1,
// DESIGN.md 2) and the quantity the conditioning guard (api.cu) bounds by kappa_max.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "setsum_mma.cuh"  // mma:: helpers (mbarrier, bulk copy, tcgen05 wrappers, smem descriptor)

namespace basq {

constexpr int NLS_NT = 256;        // candidates per tile (MMA N)
constexpr int NLS_KB = 32;         // K block (halves) per pipeline stage
constexpr int NLS_JT = 8;          // sets interleaved over a tile's columns in SETSUM mode
constexpr int NLS_A_PIECE = (NLS_KB / 8) * 128 * 16;     // 8 KB: one (landmark tile, K block) of Az hi or lo
constexpr int NLS_B_PIECE = (NLS_KB / 8) * NLS_NT * 16;  // 16 KB: one (candidate tile, K block) of kx hi or lo
constexpr int NLS_STAGE_BYTES = 2 * NLS_A_PIECE + 2 * NLS_B_PIECE;  // 48 KB
constexpr int NLS_EPI_WARPS = 8;
constexpr int NLS_THREADS = (NLS_EPI_WARPS + 3) * 32;
constexpr int NLS_KX_SHIFT = 14;   // kx operand = k / 2^ceil(log2 os) * 2^14

struct NlsDev {
  // tile geometry: slot c of tile t of set group jg <-> member e = e_lo(jg) + t * EC + c / JT of set
  // jg * JT + c % JT, local record p = set + e * S - off   (JT = 8, EC = 32: SETSUM; JT = 256, EC = 1: GRAM)
  int64_t off;
  int S;
  int64_t p_lo, p_hi;
  int jg0, n_jg;          // set groups of this chunk
  int tiles_per_jg;       // stride of the chunk's tile arrays (>= any group's tile count)
  int JT, EC;
  // operands
  const __half* azh; const __half* azl;   // [n_mtiles][KP / 8][128][8]
  const float* ainv;                      // [n_mtiles * 128] 1 / (row scale * kx scale)
  const __half* kxh; const __half* kxl;   // [n_jg * tiles_per_jg][KP / 8][256][8]
  const unsigned char* trec;              // [n_jg * tiles_per_jg][256][RB] candidate records of every tile
  int KP;                                 // padded n_obs (multiple of NLS_KB)
  const float* zz; const float* bz;       // prepared landmarks [M, DP], [M]
  const float* szf;                       // [M] per-landmark factor m(z) / mu_g(z) as fp32
  int M, n_mtiles;
  float os_f;
  double* G;
  int64_t ldg;
  double grid_m;  // reproducible instances: 1.5 * 2^52 * Q of the pass's grid Q (grid_round, common.cuh)
};

template <int DP>
struct NlsCfg {
  static constexpr int RB = ((24 + 4 * DP) + 15) / 16 * 16;
  static constexpr int REC_BYTES = NLS_NT * RB;
  static constexpr int COMB_BYTES = 2 * 128 * NLS_JT * 8;  // double-buffered hand-over of the column halves
  // operand ring as deep as shared memory allows: the stream needs 64 B/clk per SM from L2, and every stage
  // in flight hides another 768 tensor-pipe cycles of its latency (the records of a tile are single-buffered:
  // they are needed only when the tile's MMAs have finished, long after the previous tile's epilogue)
  static constexpr int FIXED = REC_BYTES + COMB_BYTES + 256;
  static constexpr int NSTAGE = (4 * NLS_STAGE_BYTES + FIXED <= 227 * 1024) ? 4 : ((3 * NLS_STAGE_BYTES + FIXED <= 227 * 1024) ? 3 : 2);
  static constexpr int OFF_STAGE = 0;
  static constexpr int OFF_REC = NSTAGE * NLS_STAGE_BYTES;
  static constexpr int OFF_COMB = OFF_REC + REC_BYTES;
  static constexpr int OFF_BAR = OFF_COMB + COMB_BYTES;
  static constexpr int SMEM_BYTES = OFF_BAR + 256;
  static_assert(SMEM_BYTES <= 227 * 1024, "nlsum: shared memory budget");
};

// member range of the JT sets from j0 that falls into [p_lo, p_hi): first member and number of tiles
__device__ __forceinline__ void nls_item_range(const NlsDev& a, int j0, int64_t& e_lo, int& n_tiles) {
  const int64_t S = a.S;
  const int64_t num_lo = a.p_lo + a.off - (int64_t)(j0 + a.JT - 1);
  e_lo = num_lo <= 0 ? 0 : (num_lo + S - 1) / S;
  const int64_t num_hi = a.p_hi - 1 + a.off - (int64_t)j0;
  const int64_t e_hi = num_hi < 0 ? 0 : num_hi / S + 1;
  const int64_t n_e = e_hi > e_lo ? e_hi - e_lo : 0;
  n_tiles = (int)((n_e + a.EC - 1) / a.EC);
}

// exact float -> double for finite floats of either sign without the conversion pipe (zero and
// denormals map to +-2^-127-sized values, far below anything the sums resolve)
__device__ __forceinline__ double f2d_signed(float v) {
  const unsigned u = __float_as_uint(v);
  return __hiloint2double((int)((((u & 0x7fffffffu) >> 3) + 0x38000000u) | (u & 0x80000000u)), (int)(u << 29));
}

// exp(c) - 1 in fp32: series below |c| < 2^-5 (relative 2e-8 there), ex2 otherwise (absolute 2e-7 e^c)
__device__ __forceinline__ float expm1_f32(float c) {
  const float e = __fsub_rn(ex2_approx(__fmul_rn(c, 1.4426950408889634f)), 1.f);
  const float p = __fmaf_rn(__fmaf_rn(__fmaf_rn(c, 0.041666668f, 0.16666667f), c, 0.5f), __fmul_rn(c, c), c);
  return fabsf(c) < 0.03125f ? p : e;
}

template <int NL>
__device__ __forceinline__ float nl_apply_f32(float c, float t) {
  if (NL == NL_WSABIM) return __fmaf_rn(__fmul_rn(0.5f, c), c, __fmul_rn(t, c));
  return __fmul_rn(t, expm1_f32(c));
}

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

// Epilogue of one 128 x 256 tile for one thread (TMEM lane = landmark row m, column half `half`):
// correction from TMEM, k(z_m, x_p) with the library's operation sequence, C, the non-linearity, fp64
// accumulation per set (MODE 0) or one store per column (MODE 1).
template <int FAM, int DP, int NL, int MODE, bool REPRO>
__device__ __forceinline__ void nls_epilogue_tile(const NlsDev& a, const unsigned char* recs, uint32_t taddr, int half,
                                                  const float (&zr)[DP], float bm, float szm, float ainv,
                                                  double (&acc)[NLS_JT], int m, bool mok, int j0) {
  constexpr int RB = NlsCfg<DP>::RB, NT = NLS_NT;
#pragma unroll 1
  for (int cb = 0; cb < NT / 2; cb += 32) {
    uint32_t v[32];
    mma::tmem_ld32(taddr + cb, v);
    mma::tmem_ld_wait();
    const int c0 = half * (NT / 2) + cb;
    double out[MODE == 1 ? 32 : 1];
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      const unsigned char* rec = recs + (c0 + c) * RB;
      const double2 hw = *reinterpret_cast<const double2*>(rec);   // per-point factor, weight
      constexpr int NF4 = (RB - 16) / 16;
      float f[NF4 * 4];                                            // [idx, a, x0, x1, ...]
#pragma unroll
      for (int q4 = 0; q4 < NF4; ++q4) {
        const float4 w4 = *reinterpret_cast<const float4*>(rec + 16 + q4 * 16);
        f[q4 * 4 + 0] = w4.x; f[q4 * 4 + 1] = w4.y; f[q4 * 4 + 2] = w4.z; f[q4 * 4 + 3] = w4.w;
      }
      const float k = pair_eval_f32<FAM, DP>(&f[2], f[1], zr, bm, a.os_f);
      const float cv = __fsub_rn(k, __fmul_rn(__uint_as_float(v[c]), ainv));
      float val = nl_apply_f32<NL>(cv, __fmul_rn(szm, (float)hw.x));
      val = (hw.y != 0.0) ? val : 0.f;
      if (MODE == 0 && REPRO) acc[c % NLS_JT] += grid_round(f2d_signed(val), hw.y, a.grid_m);
      else if (MODE == 0) acc[c % NLS_JT] = fma(f2d_signed(val), hw.y, acc[c % NLS_JT]);
      else out[c] = f2d_signed(val) * hw.y;
    }
    if (MODE == 1 && mok) {
      // one column = one cell: columns c0 .. c0 + 31 of this row are contiguous in G.  Only slots
      // that hold a candidate are written (G is zeroed by the host; a group whose members wrap
      // around the cell range spans two tiles with complementary valid slots).
      double* dst = a.G + (int64_t)m * a.ldg + j0 + c0;
#pragma unroll
      for (int c = 0; c < 32; ++c)
        if (out[c] != 0.0) dst[c] = out[c];
    }
  }
}

// MODE 0: SETSUM (accumulate per set, write once per work item) ; MODE 1: GRAM (one column = one cell)
// REPRO (MODE 0): every term is rounded to the pass's grid before it is added (see setsum_mma.cuh)
template <int FAM, int DP, int NL, int MODE, bool REPRO>
__global__ void __launch_bounds__(NLS_THREADS, 1) nlsum_kernel(const NlsDev a) {
  using Cfg = NlsCfg<DP>;
  constexpr int NSTAGE = Cfg::NSTAGE, NT = NLS_NT;
  extern __shared__ __align__(1024) unsigned char smem_nls[];
  unsigned char* const smem = smem_nls;
  unsigned char* sRec = smem + Cfg::OFF_REC;
  double* sComb = reinterpret_cast<double*>(smem + Cfg::OFF_COMB);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* s_full = bars;                 // [NSTAGE]
  uint64_t* s_empty = bars + NSTAGE;       // [NSTAGE]
  uint64_t* t_full = bars + 2 * NSTAGE;    // [2] accumulator ready
  uint64_t* t_empty = t_full + 2;          // [2] accumulator drained by the epilogue
  uint64_t* r_full = t_empty + 2;          // [1] records landed
  uint64_t* r_empty = r_full + 1;          // [1] records consumed by the epilogue
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(r_empty + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) {
      mma::mbar_init(&s_full[s], 1);
      mma::mbar_init(&s_empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mma::mbar_init(&t_full[b], 1);
      mma::mbar_init(&t_empty[b], NLS_EPI_WARPS);
    }
    mma::mbar_init(r_full, 1);
    mma::mbar_init(r_empty, NLS_EPI_WARPS);
    mma::fence_barrier_init();
  }
  if (warp == NLS_EPI_WARPS + 1) mma::tmem_alloc(tmem_slot, 512);
  mma::tc_fence_before();
  __syncthreads();
  mma::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_items = a.n_mtiles * a.n_jg;
  const int nkb = a.KP / NLS_KB;

  if (warp < NLS_EPI_WARPS) {
    // ======================================================================== epilogue
    const int quarter = warp & 3, half = warp >> 2;
    const int row = quarter * 32 + lane;          // TMEM lane = landmark row within the tile
    uint32_t tc = 0, items_done = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int mt = item % a.n_mtiles, jgl = item / a.n_mtiles;
      const int j0 = (a.jg0 + jgl) * a.JT;
      int64_t e_lo;
      int n_tiles;
      nls_item_range(a, j0, e_lo, n_tiles);
      if (n_tiles == 0) continue;
      const int m = mt * 128 + row;
      const bool mok = m < a.M;
      float zr[DP];
#pragma unroll
      for (int i = 0; i < DP; ++i) zr[i] = mok ? a.zz[(int64_t)m * DP + i] : 0.f;
      const float bm = mok ? a.bz[m] : 0.f;
      const float szm = mok ? a.szf[m] : 0.f;
      const float ainv = a.ainv[mt * 128 + row];
      double acc[NLS_JT];
#pragma unroll
      for (int jj = 0; jj < NLS_JT; ++jj) acc[jj] = 0.0;
      for (int t = 0; t < n_tiles; ++t, ++tc) {
        const uint32_t buf = tc & 1u, ph = (tc >> 1) & 1u;
        mma::mbar_wait(r_full, tc & 1u);
        mma::mbar_wait(&t_full[buf], ph);
        mma::tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * NT + half * (NT / 2);
        nls_epilogue_tile<FAM, DP, NL, MODE, REPRO>(a, sRec, taddr, half, zr, bm, szm, ainv, acc, m, mok, j0);
        mma::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mma::mbar_arrive(&t_empty[buf]);
          mma::mbar_arrive(r_empty);
        }
      }
      if (MODE == 0) {
        // combine the two column halves in a fixed order and write the item's 128 x 8 block of G
        double* comb = sComb + (items_done & 1u) * (128 * NLS_JT);
        if (half == 1) {
#pragma unroll
          for (int jj = 0; jj < NLS_JT; ++jj) comb[jj * 128 + row] = acc[jj];
        }
        mma::named_bar_sync(1, NLS_EPI_WARPS * 32);
        if (half == 0 && mok) {
          double* dst = a.G + (int64_t)m * a.ldg + j0;
#pragma unroll
          for (int jj = 0; jj < NLS_JT; ++jj)
            if (j0 + jj < a.S) dst[jj] = acc[jj] + comb[jj * 128 + row];
        }
      }
      ++items_done;
    }
  } else if (warp == NLS_EPI_WARPS) {
    // ======================================================================== operand producer
    if (lane == 0) {
      uint32_t it = 0;
      const size_t a_tile = (size_t)(a.KP / 8) * 128 * 8;   // halves per landmark tile
      const size_t b_tile = (size_t)(a.KP / 8) * NT * 8;    // halves per candidate tile
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int mt = item % a.n_mtiles, jgl = item / a.n_mtiles;
        int64_t e_lo;
        int n_tiles;
        nls_item_range(a, (a.jg0 + jgl) * a.JT, e_lo, n_tiles);
        for (int t = 0; t < n_tiles; ++t) {
          const size_t tile = (size_t)jgl * a.tiles_per_jg + t;
          for (int kb = 0; kb < nkb; ++kb, ++it) {
            const int s = it % NSTAGE;
            mma::mbar_wait(&s_empty[s], ((it / NSTAGE) & 1u) ^ 1u);
            unsigned char* st = smem + Cfg::OFF_STAGE + (size_t)s * NLS_STAGE_BYTES;
            mma::mbar_expect_tx(&s_full[s], NLS_STAGE_BYTES);
            const size_t ka = (size_t)kb * (NLS_A_PIECE / 2), kbo = (size_t)kb * (NLS_B_PIECE / 2);
            mma::bulk_g2s(st, a.azh + mt * a_tile + ka, NLS_A_PIECE, &s_full[s]);
            mma::bulk_g2s(st + NLS_A_PIECE, a.azl + mt * a_tile + ka, NLS_A_PIECE, &s_full[s]);
            mma::bulk_g2s(st + 2 * NLS_A_PIECE, a.kxh + tile * b_tile + kbo, NLS_B_PIECE, &s_full[s]);
            mma::bulk_g2s(st + 2 * NLS_A_PIECE + NLS_B_PIECE, a.kxl + tile * b_tile + kbo, NLS_B_PIECE, &s_full[s]);
          }
        }
      }
    }
  } else if (warp == NLS_EPI_WARPS + 1) {
    // ======================================================================== MMA issuer
    // instruction descriptor: D fp32 (bit 4), A / B fp16 (formats 0), K-major both, N = 256, M = 128
    constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(NT >> 3) << 17) | ((128u >> 4) << 24);
    uint32_t it = 0, tc = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int jgl = item / a.n_mtiles;
      int64_t e_lo;
      int n_tiles;
      nls_item_range(a, (a.jg0 + jgl) * a.JT, e_lo, n_tiles);
      for (int t = 0; t < n_tiles; ++t, ++tc) {
        const uint32_t buf = tc & 1u;
        mma::mbar_wait(&t_empty[buf], ((tc >> 1) & 1u) ^ 1u);
        mma::tc_fence_after();
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % NSTAGE;
          mma::mbar_wait(&s_full[s], (it / NSTAGE) & 1u);
          mma::tc_fence_after();
          if (lane == 0) {
            const uint32_t st = mma::smem_u32(smem + Cfg::OFF_STAGE + (size_t)s * NLS_STAGE_BYTES);
            const uint32_t ahi = st, alo = st + NLS_A_PIECE;
            const uint32_t bhi = st + 2 * NLS_A_PIECE, blo = bhi + NLS_B_PIECE;
            const uint32_t d = tmem_base + buf * NT;
#pragma unroll
            for (int p = 0; p < 3; ++p) {
              const uint32_t aa = (p == 0) ? alo : ahi;   // lo*hi, hi*lo, hi*hi (small terms first)
              const uint32_t bb = (p == 1) ? blo : bhi;
#pragma unroll
              for (int ks = 0; ks < NLS_KB / 16; ++ks) {
                const uint64_t ad = mma::smem_desc(aa + ks * 2 * (128 * 16), 128 * 16, 128);
                const uint64_t bd = mma::smem_desc(bb + ks * 2 * (NT * 16), NT * 16, 128);
                umma_f16(d, ad, bd, IDESC, (kb > 0 || p > 0 || ks > 0) ? 1u : 0u);
              }
            }
            mma::umma_commit(&s_empty[s]);
            if (kb == nkb - 1) mma::umma_commit(&t_full[buf]);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ======================================================================== record producer
    if (lane == 0) {
      uint32_t tc = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int jgl = item / a.n_mtiles;
        int64_t e_lo;
        int n_tiles;
        nls_item_range(a, (a.jg0 + jgl) * a.JT, e_lo, n_tiles);
        for (int t = 0; t < n_tiles; ++t, ++tc) {
          mma::mbar_wait(r_empty, (tc & 1u) ^ 1u);
          const size_t tile = (size_t)jgl * a.tiles_per_jg + t;
          mma::mbar_expect_tx(r_full, Cfg::REC_BYTES);
          mma::bulk_g2s(sRec, a.trec + tile * Cfg::REC_BYTES, Cfg::REC_BYTES, r_full);
        }
      }
    }
  }

  mma::tc_fence_before();
  __syncthreads();
  if (warp == NLS_EPI_WARPS + 1) {
    mma::tc_fence_after();
    mma::tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------
// kxgen: B operand + tile records of a chunk of set groups.  One CTA per tile, one thread per slot.
// ---------------------------------------------------------------------------------------------
struct KxDev {
  const unsigned char* recs;   // live candidate records
  int64_t off;
  int S;
  int64_t p_lo, p_hi;
  int jg0, n_jg, tiles_per_jg, JT, EC;
  const float* ozz; const float* obz;   // prepared observation "landmarks" [n_obs, DP], [n_obs]
  int n_obs, KP;
  float os_f;
  float kx_scale;                       // 2^(14 - ceil(log2 os))
  __half* kxh; __half* kxl;
  unsigned char* trec;
};

template <int FAM, int DP>
__global__ void __launch_bounds__(NLS_NT) kxgen_kernel(const KxDev a) {
  constexpr int RB = NlsCfg<DP>::RB;
  constexpr int OB = 64;                                 // observations staged per block
  __shared__ __align__(16) float s_oz[OB * DP];
  __shared__ float s_ob[OB];
  const int tile = blockIdx.x, c = threadIdx.x;
  const int jgl = tile / a.tiles_per_jg, t = tile % a.tiles_per_jg;
  const int j0 = (a.jg0 + jgl) * a.JT;
  // slot -> record
  const int64_t S = a.S;
  const int64_t num_lo = a.p_lo + a.off - (int64_t)(j0 + a.JT - 1);
  const int64_t e_lo = num_lo <= 0 ? 0 : (num_lo + S - 1) / S;
  const int ei = c / a.JT, jj = c % a.JT;
  {
    const int64_t num_hi = a.p_hi - 1 + a.off - (int64_t)j0;
    const int64_t e_hi = num_hi < 0 ? 0 : num_hi / S + 1;
    const int64_t n_e = e_hi > e_lo ? e_hi - e_lo : 0;
    if ((int64_t)t * a.EC >= n_e) return;   // beyond the group's tiles: never read (uniform over the CTA)
  }
  const int64_t e = e_lo + (int64_t)t * a.EC + ei;
  const int64_t p = (int64_t)(j0 + jj) + e * S - a.off;
  const bool ok = (j0 + jj < a.S) && (p >= a.p_lo) && (p < a.p_hi);
  float x[DP];
  float pa = 0.f;
  {
    constexpr int NV = RB / 16;
    uint4 q[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) q[v] = make_uint4(0u, 0u, 0u, 0u);
    if (ok) {
      const uint4* rec = reinterpret_cast<const uint4*>(a.recs + p * RB);
#pragma unroll
      for (int v = 0; v < NV; ++v) q[v] = __ldg(rec + v);
    }
    uint4* dst = reinterpret_cast<uint4*>(a.trec + ((size_t)tile * NLS_NT + c) * RB);
#pragma unroll
    for (int v = 0; v < NV; ++v) dst[v] = q[v];           // invalid slots: all zero (weight 0, finite coordinates)
    float f[(NV - 1) * 4];
#pragma unroll
    for (int v = 1; v < NV; ++v) {
      f[(v - 1) * 4 + 0] = __uint_as_float(q[v].x);
      f[(v - 1) * 4 + 1] = __uint_as_float(q[v].y);
      f[(v - 1) * 4 + 2] = __uint_as_float(q[v].z);
      f[(v - 1) * 4 + 3] = __uint_as_float(q[v].w);
    }
    pa = f[1];
#pragma unroll
    for (int i = 0; i < DP; ++i) x[i] = f[2 + i];
  }
  const size_t b_tile = (size_t)(a.KP / 8) * NLS_NT * 8;
  uint4* oh = reinterpret_cast<uint4*>(a.kxh + (size_t)tile * b_tile) + c;
  uint4* ol = reinterpret_cast<uint4*>(a.kxl + (size_t)tile * b_tile) + c;
  for (int o0 = 0; o0 < a.KP; o0 += OB) {
    __syncthreads();
    for (int i = threadIdx.x; i < OB * DP; i += NLS_NT) {
      const int o = o0 + i / DP;
      s_oz[i] = o < a.n_obs ? a.ozz[(size_t)o * DP + i % DP] : 0.f;
    }
    if (threadIdx.x < OB) s_ob[threadIdx.x] = (o0 + (int)threadIdx.x < a.n_obs) ? a.obz[o0 + threadIdx.x] : 0.f;
    __syncthreads();
    const int ob_end = min(OB, a.KP - o0);
    for (int kc = 0; kc < ob_end / 8; ++kc) {
      __half2 h2[4], l2[4];
#pragma unroll
      for (int u = 0; u < 8; u += 2) {
        float vv[2];
#pragma unroll
        for (int w = 0; w < 2; ++w) {
          const int ol_ = kc * 8 + u + w;
          float kv = 0.f;
          if (ok && o0 + ol_ < a.n_obs) kv = pair_eval_f32<FAM, DP>(x, pa, &s_oz[ol_ * DP], s_ob[ol_], a.os_f);
          vv[w] = __fmul_rn(kv, a.kx_scale);
        }
        const __half h0 = __float2half_rn(vv[0]), h1 = __float2half_rn(vv[1]);
        h2[u / 2] = __halves2half2(h0, h1);
        l2[u / 2] = __halves2half2(__float2half_rn(__fsub_rn(vv[0], __half2float(h0))),
                                   __float2half_rn(__fsub_rn(vv[1], __half2float(h1))));
      }
      const size_t chunk = (size_t)(o0 / 8 + kc) * NLS_NT;
      oh[chunk] = *reinterpret_cast<const uint4*>(h2);
      ol[chunk] = *reinterpret_cast<const uint4*>(l2);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// fp64 matrix -> row-scaled fp16 hi / lo operand tiles (Az here, T = tril(W + W^T) in gpvar.cuh)
// ---------------------------------------------------------------------------------------------
// REV (square A, rows == cols == n): the operand is the lower triangle of J G^T J, J the reversal
// permutation - element [m, o] is G[n-1-o, n-1-m] for o <= m and 0 above the diagonal; G's upper
// triangle is never read.  L^-1 of a GP comes out of the Cholesky factor G of J W J in this form (gpvar.cu).
template <bool REV>
__device__ __forceinline__ double op16_at(const double* __restrict__ A, int rows, int64_t lda, int m, int o) {
  if (!REV) return A[(int64_t)m * lda + o];
  return o <= m ? A[(int64_t)(rows - 1 - o) * lda + (rows - 1 - m)] : 0.0;
}

// one block per row: r = 2^(13 - floor(log2 max_o |A[m, o]|)), so that the scaled row lies in [2^13, 2^14);
// inv[m] = 1 / (r * kx_scale) (a power of two, exact).  Rows beyond `rows` get 0.
template <int THREADS, bool REV = false>
__global__ void rowscale16_kernel(const double* __restrict__ A, int rows, int cols, int64_t lda, float kx_scale,
                                  float* __restrict__ rscale, float* __restrict__ inv) {
  __shared__ double sh[THREADS];
  const int m = blockIdx.x;
  double mx = 0.0;
  if (m < rows)
    for (int o = threadIdx.x; o < (REV ? m + 1 : cols); o += THREADS) mx = fmax(mx, fabs(op16_at<REV>(A, rows, lda, m, o)));
  sh[threadIdx.x] = mx;
  __syncthreads();
  for (int w = THREADS / 2; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + w]);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    float r = 0.f, iv = 0.f;
    if (m < rows) {
      int e = 0;
      if (sh[0] > 0.0 && isfinite(sh[0])) e = 13 - ilogb(sh[0]);
      e = max(-40, min(40, e));  // a row this small contributes nothing; keep every factor a normal float
      r = ldexpf(1.f, e);
      iv = 1.f / (r * kx_scale);
    }
    rscale[m] = r;
    inv[m] = iv;
  }
}

// one thread per (row tile, K chunk of 8, row): 8 scaled values -> fp16 hi / lo, 16-byte stores into
// [tile][KP / 8][TILE_ROWS][8 halves]
template <int TILE_ROWS, bool REV = false>
__global__ void split16_kernel(const double* __restrict__ A, int rows, int cols, int64_t lda, int KP, int n_tiles,
                               const float* __restrict__ rscale, __half* __restrict__ hi, __half* __restrict__ lo) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int KC = KP / 8;
  if (t >= (int64_t)n_tiles * KC * TILE_ROWS) return;
  const int r = (int)(t % TILE_ROWS);
  const int kc = (int)((t / TILE_ROWS) % KC);
  const int mt = (int)(t / (TILE_ROWS * (int64_t)KC));
  const int m = mt * TILE_ROWS + r;
  __half h[8], l[8];
  const double rs = m < rows ? (double)rscale[m] : 0.0;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int o = kc * 8 + e;
    const double x = (m < rows && o < cols) ? op16_at<REV>(A, rows, lda, m, o) * rs : 0.0;
    h[e] = __double2half(x);
    l[e] = __double2half(x - (double)__half2float(h[e]));   // residual against the fp64 value: ~22 bits in hi + lo
  }
  reinterpret_cast<uint4*>(hi)[t] = *reinterpret_cast<const uint4*>(h);
  reinterpret_cast<uint4*>(lo)[t] = *reinterpret_cast<const uint4*>(l);
}

// launchers, one translation unit per (family, non-linearity): nlsum_inst_*.cu
template <int FAM, int DP, int NL>
int launch_nlsum_dp(basq_ctx* ctx, const NlsDev& dev, int mode) {
  using Cfg = NlsCfg<DP>;
  BASQ_CHECK((size_t)Cfg::SMEM_BYTES <= ctx->smem_optin, BASQ_ERR_UNSUPPORTED,
             "nlsum: kernel needs %d B shared memory (limit %zu)", Cfg::SMEM_BYTES, ctx->smem_optin);
  const int64_t n_items = (int64_t)dev.n_mtiles * dev.n_jg;
  const int grid = (int)std::min<int64_t>(ctx->num_sms, n_items);
  if (grid <= 0) return BASQ_OK;
  if (mode == 0 && dev.grid_m != 0.0) {
    BASQ_CUDA(cudaFuncSetAttribute(nlsum_kernel<FAM, DP, NL, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    nlsum_kernel<FAM, DP, NL, 0, true><<<grid, NLS_THREADS, Cfg::SMEM_BYTES, ctx->stream>>>(dev);
  } else if (mode == 0) {
    BASQ_CUDA(cudaFuncSetAttribute(nlsum_kernel<FAM, DP, NL, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    nlsum_kernel<FAM, DP, NL, 0, false><<<grid, NLS_THREADS, Cfg::SMEM_BYTES, ctx->stream>>>(dev);
  } else {
    BASQ_CUDA(cudaFuncSetAttribute(nlsum_kernel<FAM, DP, NL, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    nlsum_kernel<FAM, DP, NL, 1, false><<<grid, NLS_THREADS, Cfg::SMEM_BYTES, ctx->stream>>>(dev);
  }
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

template <int FAM, int NL>
int launch_nlsum_family(basq_ctx* ctx, int dp, const NlsDev& dev, int mode) {
  switch (dp) {
    case 2: return launch_nlsum_dp<FAM, 2, NL>(ctx, dev, mode);
    case 4: return launch_nlsum_dp<FAM, 4, NL>(ctx, dev, mode);
    case 6: return launch_nlsum_dp<FAM, 6, NL>(ctx, dev, mode);
    case 8: return launch_nlsum_dp<FAM, 8, NL>(ctx, dev, mode);
    case 10: return launch_nlsum_dp<FAM, 10, NL>(ctx, dev, mode);
    case 12: return launch_nlsum_dp<FAM, 12, NL>(ctx, dev, mode);
    case 16: return launch_nlsum_dp<FAM, 16, NL>(ctx, dev, mode);
    case 20: return launch_nlsum_dp<FAM, 20, NL>(ctx, dev, mode);
    case 24: return launch_nlsum_dp<FAM, 24, NL>(ctx, dev, mode);
    case 32: return launch_nlsum_dp<FAM, 32, NL>(ctx, dev, mode);
  }
  set_error("nlsum: no kernel compiled for padded dimension %d", dp);
  return BASQ_ERR_UNSUPPORTED;
}

template <int FAM, int DP>
int launch_kxgen_dp(basq_ctx* ctx, const KxDev& dev) {
  const int64_t tiles = (int64_t)dev.n_jg * dev.tiles_per_jg;
  if (tiles <= 0) return BASQ_OK;
  kxgen_kernel<FAM, DP><<<(unsigned)tiles, NLS_NT, 0, ctx->stream>>>(dev);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

template <int FAM>
int launch_kxgen_family(basq_ctx* ctx, int dp, const KxDev& dev) {
  switch (dp) {
    case 2: return launch_kxgen_dp<FAM, 2>(ctx, dev);
    case 4: return launch_kxgen_dp<FAM, 4>(ctx, dev);
    case 6: return launch_kxgen_dp<FAM, 6>(ctx, dev);
    case 8: return launch_kxgen_dp<FAM, 8>(ctx, dev);
    case 10: return launch_kxgen_dp<FAM, 10>(ctx, dev);
    case 12: return launch_kxgen_dp<FAM, 12>(ctx, dev);
    case 16: return launch_kxgen_dp<FAM, 16>(ctx, dev);
    case 20: return launch_kxgen_dp<FAM, 20>(ctx, dev);
    case 24: return launch_kxgen_dp<FAM, 24>(ctx, dev);
    case 32: return launch_kxgen_dp<FAM, 32>(ctx, dev);
  }
  set_error("kxgen: no kernel compiled for padded dimension %d", dp);
  return BASQ_ERR_UNSUPPORTED;
}

// fam in {RBF, MATERN15, MATERN25}, nl in {NL_WSABIM, NL_MMLT}
int launch_nlsum(basq_ctx* ctx, int fam, int nl, int dp, const NlsDev& dev, int mode);
int launch_kxgen(basq_ctx* ctx, int fam, int dp, const KxDev& dev);
int launch_nlsum_rbf_wm(basq_ctx*, int, const NlsDev&, int);
int launch_nlsum_rbf_ml(basq_ctx*, int, const NlsDev&, int);
int launch_nlsum_m15_wm(basq_ctx*, int, const NlsDev&, int);
int launch_nlsum_m15_ml(basq_ctx*, int, const NlsDev&, int);
int launch_nlsum_m25_wm(basq_ctx*, int, const NlsDev&, int);
int launch_nlsum_m25_ml(basq_ctx*, int, const NlsDev&, int);
int launch_kxgen_rbf(basq_ctx*, int, const KxDev&);
int launch_kxgen_m15(basq_ctx*, int, const KxDev&);
int launch_kxgen_m25(basq_ctx*, int, const KxDev&);

}  // namespace basq
