// Caratheodory step, register-resident block-pivot version (the fast path; car.cu keeps the general
// global-memory kernel for shapes beyond its limits).  Same algorithm as car.cu:
//   stage 1  Gauss-Jordan with row pivoting turns A [n, S] into [I | T]      (null-space basis)
//   stage 2  ratio-test eliminations of the m = S - n non-basic sets          (BASQ/_rchq.py:146-171)
//
// The step is a chain of n + m strictly sequential pivots: what matters is the latency of ONE pivot.
// B200 mapping.  One persistent cooperative kernel, NT threads per CTA, one CTA per SM.
//   * The tableau never touches shared or global memory between pivots: CTA k keeps a block of B
//     consecutive rows (stage 1) / non-basic columns (stage 2) in REGISTERS, thread t holding the
//     entries of columns (rows) t, t+NT, t+2NT, ... of each of them.
//   * The owner CTA performs its B pivots back to back on its own registers with ONE __syncthreads
//     per pivot: the block arg-reduce carries, next to the winner's key, the B multipliers of its
//     column (stage 1) / row (stage 2) and the correctly rounded reciprocal of its pivot, which
//     every lane computes for its own candidate ahead of the reduction; sibling updates are
//     register FMAs.
//   * Publication is "the data is the flag": the pivot row (column) and a per-thread copy of the
//     pivot index are streamed to L2 buffers that the host pre-filled with a NaN / -1 sentinel; a
//     consumer thread simply polls the few words IT needs until they are no longer the sentinel.
//     No fences, no flags, no grid barrier on the pivot chain (one barrier between the stages):
//     consumers replay pivot i while the owner is already working on pivot i+1, so the chain per
//     block is the owner's B pivots + one L2 round trip + ONE replayed pivot of the next owner.
//   * Stage 2 hands the basic weights from owner to owner the same way; CTAs whose columns are
//     eliminated exit.
// Limits: S <= CPT*NT = 2048, n <= RPT*NT = 1024, n, m <= 8 * #SMs.
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "gridsync.cuh"

namespace basq {

namespace {

constexpr unsigned FULLMASK = 0xffffffffu;

struct Car2Dev {
  double* A;
  int n, S;
  int64_t lda;
  double* prow;     // [n][S]      pivot rows as published (NaN-sentinel filled)
  int* prep;        // [n][NT]     per-thread copies of the row's pivot code (-1 = not yet published)
  int* pinfo;       // [n]         pivot column of row r, -1 = row skipped (dependent)
  double* pcol;     // [S][n]      pivot columns as published (stage 2; NaN-sentinel filled)
  int* srep;        // [S][NT]     per-thread copies of the column's leaving-row code
  double* muh;      // [G2][n]     basic weights handed to the owner of block k+1 (NaN-sentinel filled)
  int* rph;         // [G2][n]     row -> set map handed over (code = set + 2)
  double* omega;    // [S]
  unsigned* bar;
  int* status;
  unsigned long long* stamps;  // optional [4] globaltimer stamps (BASQ_CAR_TIMING=1): start, stage 1 done, barrier passed, end
  double tol;
};

__device__ __forceinline__ void stamp(unsigned long long* stamps, int i) {
  if (stamps) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    stamps[i] = t;
  }
}

// pivot codes: -1 not published, 1 = none (row skipped / no basic set leaves), c + 2 = index c
// (is_sentinel / poll_f64 / poll_i32: gridsync.cuh)

// ---------------------------------------------------------------------------------------------
// Block-wide arg-max / arg-min with ONE barrier.
// The key is a non-negative double, so its bit pattern orders like an unsigned integer; the low 12
// mantissa bits are replaced by the candidate's index (complemented for the maximum), which makes
// every candidate unique and breaks ties (keys equal to 2^-40 relative) towards the smaller index.
// The winner's exact payload (W words: signed pivot / exact ratio, reciprocal, multipliers) travels
// through the scratch slots: the lane that recognises its own packed key as the warp's best writes
// its key and calls fill(payload row), and after the barrier every warp reduces the NT/32 warp keys
// itself and reads the global winner's payload row.
// The slots are double-buffered by the CTA-uniform parity spar, and every read of the slots of call
// N (keys, and the payload words the caller reads before its next call) happens before the reading
// thread arrives at the barrier of call N+1.  A thread writes the same parity again only in call
// N+2, after passing that barrier, i.e. after every thread has finished reading call N.
// ---------------------------------------------------------------------------------------------
template <int NT, int W>
struct Scratch {
  static_assert(W % 2 == 0, "payload rows stay 16-byte aligned");
  unsigned long long key[2][NT / 32];
  alignas(16) double pay[2][NT / 32][W];
};

__device__ __forceinline__ unsigned long long pack_max(double key, int idx) {
  return ((unsigned long long)__double_as_longlong(key) & ~0xFFFull) | (unsigned long long)(0xFFF - idx);
}
__device__ __forceinline__ unsigned long long pack_min(double key, int idx) {
  return ((unsigned long long)__double_as_longlong(key) & ~0xFFFull) | (unsigned long long)idx;
}
// 64-bit max / min over a warp with the integer reduction unit: two REDUX (high words, then the low
// words of the lanes that tie on the high word) instead of a five-round 64-bit shuffle butterfly.
template <bool MAX>
__device__ __forceinline__ unsigned long long warp_best_u64(unsigned long long x) {
  const unsigned hi = (unsigned)(x >> 32), lo = (unsigned)x;
  if (MAX) {
    const unsigned mhi = __reduce_max_sync(FULLMASK, hi);
    const unsigned mlo = __reduce_max_sync(FULLMASK, hi == mhi ? lo : 0u);
    return ((unsigned long long)mhi << 32) | mlo;
  } else {
    const unsigned mhi = __reduce_min_sync(FULLMASK, hi);
    const unsigned mlo = __reduce_min_sync(FULLMASK, hi == mhi ? lo : 0xFFFFFFFFu);
    return ((unsigned long long)mhi << 32) | mlo;
  }
}

template <bool MAX>
__device__ __forceinline__ int key_index(unsigned long long key) {
  return MAX ? (0xFFF - (int)(key & 0xFFFull)) : (int)(key & 0xFFFull);
}

// Returns the winner's index (-1: no candidate; MAX: `none` = 0, MIN: `none` = ~0) and points `pay`
// at its payload row (valid only for a winner).
template <bool MAX, int NT, int W, class Fill>
__device__ __forceinline__ int block_best(unsigned long long mine, Scratch<NT, W>& s, int& spar, const double*& pay,
                                          Fill fill) {
  constexpr unsigned long long NONE = MAX ? 0ull : ~0ull;
  const unsigned long long x = warp_best_u64<MAX>(mine);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (x == NONE) {
    if (lane == 0) s.key[spar][warp] = NONE;
  } else if (mine == x) {
    s.key[spar][warp] = x;
    fill(s.pay[spar][warp]);
  }
  __syncthreads();
  const int p = spar;
  spar ^= 1;
  const unsigned long long w = s.key[p][lane & (NT / 32 - 1)];
  const unsigned long long y = warp_best_u64<MAX>(w);
  const unsigned hit = __ballot_sync(FULLMASK, w == y);
  pay = s.pay[p][(__ffs(hit) - 1) & (NT / 32 - 1)];
  return y == NONE ? -1 : key_index<MAX>(y);
}

template <int B, int NT, int CPT, int RPT>
__global__ void __launch_bounds__(NT, 1) car2_kernel(const Car2Dev a) {
  // payload row: stage 1 {B multipliers, reciprocal of the pivot}, stage 2 {B multipliers, ratio}
  constexpr int W = (B + 2) & ~1;
  __shared__ Scratch<NT, W> scratch;
  __shared__ double fbuf[2][B];
  __shared__ int abort_sh;
  extern __shared__ int nbcol[];  // [S] non-basic column list (stage 2)

  const int n = a.n, S = a.S;
  const int G = gridDim.x, b = blockIdx.x, tid = threadIdx.x;
  unsigned gen = 0;
  int par = 0;   // parity of the multiplier buffer (advanced once per applied pivot, CTA-uniform)
  int spar = 0;  // parity of the arg-reduce scratch

  for (int c = b * NT + tid; c < S; c += G * NT) a.omega[c] = 0.0;
  if (b == 0 && tid == 0) stamp(a.stamps, 0);

  // ------------------------------------------------------------------ stage 1: own rows -> registers
  const int G1 = (n + B - 1) / B;
  const int r0 = b * B;
  const int rows_mine = max(0, min(B, n - r0));
  double reg[B][CPT];
  // largest |entry| of each own row (CTA-uniform; in shared memory, which keeps B = 8 free of spills at
  // 128 registers).  Thread 0 writes it; the barrier of the next block_best publishes it.
  __shared__ double rscale[B];
  unsigned elig = 0;
#pragma unroll
  for (int j = 0; j < CPT; ++j)
    if (tid + j * NT < S) elig |= 1u << j;
#pragma unroll
  for (int i = 0; i < B; ++i) {
#pragma unroll
    for (int j = 0; j < CPT; ++j) {
      const int c = tid + j * NT;
      reg[i][j] = (i < rows_mine && c < S) ? a.A[(int64_t)(r0 + i) * a.lda + c] : 0.0;
    }
  }
#pragma unroll
  for (int i = 0; i < B; ++i) {
    unsigned long long mk = 0ull;
    double mv = 0.0;
    if (i < rows_mine) {
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        const unsigned long long pk = pack_max(fabs(reg[i][j]), tid + j * NT);
        if ((elig >> j & 1u) && pk > mk) { mk = pk; mv = reg[i][j]; }
      }
    }
    const double* w;
    const int idx = block_best<true>(mk, scratch, spar, w, [&](double* p) { p[0] = mv; });
    if (tid == 0) rscale[i] = idx < 0 ? 0.0 : fabs(w[0]);  // (CTA-uniform loop: every thread calls it B times)
  }

  // Rows and columns past the own block (rows_mine < B, cols_mine < B: a ragged last block or an
  // idle CTA) start at zero, receive the same updates as the others and are never read: no
  // predicates for them in the updates below.
  // Consumer replay: rank-1 update of the own rows with pivot-row entries `pr` (pivot column cs);
  // the thread holding column cs broadcasts its B multipliers through fbuf.
  auto eliminate = [&](const double (&pr)[CPT], int cs) {
    const bool holder = (cs & (NT - 1)) == tid;
    const int js = cs / NT;
    if (holder) {
      elig &= ~(1u << js);
#pragma unroll
      for (int j = 0; j < CPT; ++j)
        if (j == js) {
#pragma unroll
          for (int i2 = 0; i2 < B; ++i2) fbuf[par][i2] = reg[i2][j];
        }
    }
    __syncthreads();
#pragma unroll
    for (int i2 = 0; i2 < B; ++i2) {
      const double f = fbuf[par][i2];
#pragma unroll
      for (int j = 0; j < CPT; ++j) reg[i2][j] = fma(-f, pr[j], reg[i2][j]);
    }
    if (holder) {  // the eliminated column is exactly zero in every other row
#pragma unroll
      for (int j = 0; j < CPT; ++j)
        if (j == js) {
#pragma unroll
          for (int i2 = 0; i2 < B; ++i2) reg[i2][j] = 0.0;
        }
    }
    par ^= 1;
  };

  for (int k = 0; k < G1; ++k) {
    const int kr0 = k * B;
    const int krows = min(B, n - kr0);
    if (b == k) {
      // ---- owner: B local pivots, each published as soon as it exists
      if (tid == 0 && (b == 10 || b == 11)) stamp(a.stamps, b == 10 ? 4 : 6);
#pragma unroll
      for (int i = 0; i < B; ++i) {
        if (i < krows) {
          unsigned long long mk = 0ull;
          double mv = 0.0;
#pragma unroll
          for (int j = 0; j < CPT; ++j) {
            const unsigned long long pk = pack_max(fabs(reg[i][j]), tid + j * NT);
            if ((elig >> j & 1u) && pk > mk) { mk = pk; mv = reg[i][j]; }
          }
          // every lane inverts its own candidate while the reduction runs (1 avoids the slow path
          // for lanes without one; a zero pivot is skipped below and its reciprocal never used)
          const double rinv = __drcp_rn(mv != 0.0 ? mv : 1.0);
          const double* w;
          // payload: the PRE-scaling entries of the candidate column in all B rows (the sibling
          // multipliers; entry i is the pivot itself) and the reciprocal of the pivot
          const int cs = block_best<true>(mk, scratch, spar, w, [&](double* p) {
            const int jm = key_index<true>(mk) / NT;
#pragma unroll
            for (int j = 0; j < CPT; ++j)
              if (j == jm) {
#pragma unroll
                for (int i2 = 0; i2 < B; ++i2) p[i2] = reg[i2][j];
              }
            p[B] = rinv;
          });
          const bool skip = (cs < 0) || !(fabs(w[i]) > a.tol * rscale[i]) || !(rscale[i] > 0.0);
          const int row = kr0 + i;
          if (skip) {
            __stcg(&a.prep[(int64_t)row * NT + tid], 1);
            if (tid == 0) a.pinfo[row] = -1;
          } else {
            const double inv = w[B];
#pragma unroll
            for (int j = 0; j < CPT; ++j) reg[i][j] = (tid + j * NT == cs) ? 1.0 : reg[i][j] * inv;
            // the next pivot's row first, then the other siblings, then the publication stores
#pragma unroll
            for (int s = 1; s < B; ++s) {
              const int i2 = (i + s) % B;
              const double f = w[i2];
#pragma unroll
              for (int j = 0; j < CPT; ++j) reg[i2][j] = fma(-f, reg[i][j], reg[i2][j]);
            }
            if ((cs & (NT - 1)) == tid) {  // the eliminated column is exactly zero in every other row
              const int js = cs / NT;
              elig &= ~(1u << js);
#pragma unroll
              for (int j = 0; j < CPT; ++j)
                if (j == js) {
#pragma unroll
                  for (int i2 = 0; i2 < B; ++i2)
                    if (i2 != i) reg[i2][j] = 0.0;
                }
            }
#pragma unroll
            for (int j = 0; j < CPT; ++j) {
              const int c = tid + j * NT;
              if (c < S) __stcg(&a.prow[(int64_t)row * S + c], reg[i][j]);
            }
            __stcg(&a.prep[(int64_t)row * NT + tid], cs + 2);
            if (tid == 0) a.pinfo[row] = cs;
          }
        }
      }
      if (tid == 0 && b == 10) stamp(a.stamps, 5);
    } else {
      // ---- everyone else: replay the block's rank-1 updates as the pivots appear in L2 (codes of the
      // whole block and a rolling window of pivot-row entries are requested ahead of use)
      int code[B];
#pragma unroll
      for (int i = 0; i < B; ++i) code[i] = (i < krows) ? __ldcg(&a.prep[(int64_t)(kr0 + i) * NT + tid]) : 1;
      constexpr int PF = (B < 3) ? B : 3;
      double win[PF][CPT];
#pragma unroll
      for (int i = 0; i < PF; ++i)
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
          const int c = tid + j * NT;
          win[i][j] = (i < krows && c < S) ? __ldcg(&a.prow[(int64_t)(kr0 + i) * S + c]) : 0.0;
        }
#pragma unroll
      for (int i = 0; i < B; ++i) {
        if (i < krows) {
          // Wait until pivot i is complete in registers.  Every missing word of pivots i .. i+PF-1 is
          // re-requested in ONE batch of independent loads per round trip (a chain of dependent
          // polls would cost one L2 round trip per word).
          for (int spins = 0;; ++spins) {
            bool ok = code[i] != -1;
            if (code[i] >= 2) {
#pragma unroll
              for (int j = 0; j < CPT; ++j)
                if (tid + j * NT < S && is_sentinel(win[i % PF][j])) ok = false;
            }
            if (ok) break;
            if ((spins & 63) == 63 && (*reinterpret_cast<volatile int*>(a.status) != 0 || spins > BASQ_SPIN_LIMIT)) {
              if (spins > BASQ_SPIN_LIMIT) atomicExch(a.status, 2);
              code[i] = 1;
              break;
            }
#pragma unroll
            for (int w = 0; w < PF; ++w) {
              if (i + w < B && i + w < krows) {
                if (code[i + w] == -1) code[i + w] = __ldcg(&a.prep[(int64_t)(kr0 + i + w) * NT + tid]);
#pragma unroll
                for (int j = 0; j < CPT; ++j) {
                  const int c = tid + j * NT;
                  if (c < S && is_sentinel(win[(i + w) % PF][j]))
                    win[(i + w) % PF][j] = __ldcg(&a.prow[(int64_t)(kr0 + i + w) * S + c]);
                }
              }
            }
          }
          const int cd = code[i];
          double cur[CPT];
#pragma unroll
          for (int j = 0; j < CPT; ++j) {
            cur[j] = win[i % PF][j];
            const int c = tid + j * NT;
            if (i + PF < B) win[i % PF][j] = (i + PF < krows && c < S) ? __ldcg(&a.prow[(int64_t)(kr0 + i + PF) * S + c]) : 0.0;
          }
          if (cd >= 2) eliminate(cur, cd - 2);
        }
      }
    }
  }

  if (b == G1 - 1 && tid == 0) stamp(a.stamps, 1);
  // ------------------------------------------------------------------ write [I | T] back, list the non-basic sets
#pragma unroll
  for (int i = 0; i < B; ++i)
    if (i < rows_mine) {
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        const int c = tid + j * NT;
        if (c < S) __stcg(&a.A[(int64_t)(r0 + i) * a.lda + c], reg[i][j]);
      }
    }
  // ascending list of still-eligible (= non-basic) columns: warp ballots + a scan over the warp counts
  __shared__ int wcnt[CPT][NT / 32];
  __shared__ int m_sh;
  {
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int j = 0; j < CPT; ++j) {
      const unsigned mask = __ballot_sync(FULLMASK, (elig >> j) & 1u);
      if (lane == 0) wcnt[j][warp] = __popc(mask);
    }
    __syncthreads();
    int base = 0;
#pragma unroll
    for (int j = 0; j < CPT; ++j) {
      int before = 0, total = 0;
      for (int w = 0; w < NT / 32; ++w) {
        const int cnt = wcnt[j][w];
        if (w < warp) before += cnt;
        total += cnt;
      }
      const unsigned mask = __ballot_sync(FULLMASK, (elig >> j) & 1u);
      if ((elig >> j) & 1u) nbcol[base + before + __popc(mask & ((1u << lane) - 1u))] = tid + j * NT;
      base += total;
    }
    if (tid == 0) m_sh = base;
    __syncthreads();
  }
  const int m = m_sh;
  if ((m + B - 1) / B > G) {
    // more non-basic sets than this launch can hold in registers (rank-deficient system):
    // tell the host to redo the step with the general kernel.  Uniform over the grid.
    if (b == 0 && tid == 0) atomicExch(a.status, 3);
    return;
  }
  if (grid_barrier(a.bar, gen, a.status, &abort_sh)) return;
  if (b == 0 && tid == 0) stamp(a.stamps, 2);

  // ------------------------------------------------------------------ stage 2: own non-basic columns -> registers
  const int G2 = (m + B - 1) / B;
  if (b >= G2) return;  // no columns here; nobody waits for this CTA
  const int c0 = b * B;
  const int cols_mine = max(0, min(B, m - c0));
  double tc[B][RPT];
  double muB[RPT];
  int rowpt[RPT];
#pragma unroll
  for (int jj = 0; jj < RPT; ++jj) {
    const int i = tid + jj * NT;
    rowpt[jj] = (i < n) ? __ldcg(&a.pinfo[i]) : -1;
    muB[jj] = (rowpt[jj] >= 0) ? 1.0 : 0.0;
  }
#pragma unroll
  for (int l = 0; l < B; ++l) {
#pragma unroll
    for (int jj = 0; jj < RPT; ++jj) {
      const int i = tid + jj * NT;
      tc[l][jj] = (l < cols_mine && i < n && rowpt[jj] >= 0) ? __ldcg(&a.A[(int64_t)i * a.lda + nbcol[c0 + l]]) : 0.0;
    }
  }

  // consumer replay: pivot the own columns on basic row istar of the published column pv; the
  // thread holding row istar broadcasts the B multipliers through fbuf
  auto col_update = [&](const double (&pv)[RPT], int istar) {
    const bool holder = (istar & (NT - 1)) == tid;
    const int js = istar / NT;
    if (holder) {
#pragma unroll
      for (int jj = 0; jj < RPT; ++jj)
        if (jj == js) {
          const double invp = __drcp_rn(pv[jj]);
#pragma unroll
          for (int l2 = 0; l2 < B; ++l2) fbuf[par][l2] = tc[l2][jj] * invp;
        }
    }
    __syncthreads();
#pragma unroll
    for (int l2 = 0; l2 < B; ++l2) {
      const double t = fbuf[par][l2];
#pragma unroll
      for (int jj = 0; jj < RPT; ++jj) tc[l2][jj] = fma(-pv[jj], t, tc[l2][jj]);
    }
    if (holder) {  // the leaving row holds the multiplier itself
#pragma unroll
      for (int jj = 0; jj < RPT; ++jj)
        if (jj == js) {
#pragma unroll
          for (int l2 = 0; l2 < B; ++l2) tc[l2][jj] = fbuf[par][l2];
        }
    }
    par ^= 1;
  };

  for (int k = 0; k <= b; ++k) {
    const int kc0 = k * B;
    const int kcols = min(B, m - kc0);
    if (k < b) {
      // ---- replay the block's pivots on the own columns as they appear
      int code[B];
      double pvs[B][RPT];
#pragma unroll
      for (int l = 0; l < B; ++l) {
        code[l] = (l < kcols) ? __ldcg(&a.srep[(int64_t)(kc0 + l) * NT + tid]) : 1;
#pragma unroll
        for (int jj = 0; jj < RPT; ++jj) {
          const int i = tid + jj * NT;
          pvs[l][jj] = (l < kcols && i < n) ? __ldcg(&a.pcol[(int64_t)(kc0 + l) * n + i]) : 0.0;
        }
      }
#pragma unroll
      for (int l = 0; l < B; ++l) {
        if (l < kcols) {
          // as in stage 1: all missing words of pivots l .. B-1 in one batch of loads per round trip
          for (int spins = 0;; ++spins) {
            bool ok = code[l] != -1;
            if (code[l] >= 2) {
#pragma unroll
              for (int jj = 0; jj < RPT; ++jj)
                if (tid + jj * NT < n && is_sentinel(pvs[l][jj])) ok = false;
            }
            if (ok) break;
            if ((spins & 63) == 63 && (*reinterpret_cast<volatile int*>(a.status) != 0 || spins > BASQ_SPIN_LIMIT)) {
              if (spins > BASQ_SPIN_LIMIT) atomicExch(a.status, 2);
              code[l] = 1;
              break;
            }
#pragma unroll
            for (int l2 = l; l2 < B; ++l2) {
              if (l2 < kcols) {
                if (code[l2] == -1) code[l2] = __ldcg(&a.srep[(int64_t)(kc0 + l2) * NT + tid]);
#pragma unroll
                for (int jj = 0; jj < RPT; ++jj) {
                  const int i = tid + jj * NT;
                  if (i < n && is_sentinel(pvs[l2][jj])) pvs[l2][jj] = __ldcg(&a.pcol[(int64_t)(kc0 + l2) * n + i]);
                }
              }
            }
          }
          if (code[l] >= 2) col_update(pvs[l], code[l] - 2);
        }
      }
    } else {
      // ---- owner: take over the basic weights, then its columns' ratio tests (reference :148-159)
      if (k > 0) {
#pragma unroll
        for (int jj = 0; jj < RPT; ++jj) {
          const int i = tid + jj * NT;
          if (i < n) {
            rowpt[jj] = poll_i32(&a.rph[(int64_t)(k - 1) * n + i], a.status) - 2;
            muB[jj] = poll_f64(&a.muh[(int64_t)(k - 1) * n + i], a.status);
          }
        }
      }
#pragma unroll
      for (int l = 0; l < B; ++l) {
        if (l < kcols) {
          unsigned long long bk = ~0ull;
          double bv = 0.0, bt = -1.0;  // (-1: no candidate; keeps the reciprocal off its slow path)
#pragma unroll
          for (int jj = 0; jj < RPT; ++jj) {
            const double t = tc[l][jj];
            if (rowpt[jj] >= 0 && t < 0.0) {
              const double ratio = muB[jj] / (-t);
              const unsigned long long pk = pack_min(ratio, tid + jj * NT);
              if (pk < bk) { bk = pk; bv = ratio; bt = t; }
            }
          }
          const double rinvp = __drcp_rn(bt);  // computed by every lane while the reduction runs
          const double* w;
          // payload: the multipliers of the later own columns (entries of the candidate row scaled
          // by the reciprocal of the pivot) and the ratio
          const int best = block_best<false>(bk, scratch, spar, w, [&](double* p) {
            const int jm = key_index<false>(bk) / NT;
#pragma unroll
            for (int jj = 0; jj < RPT; ++jj)
              if (jj == jm) {
#pragma unroll
                for (int l2 = l + 1; l2 < B; ++l2) p[l2] = tc[l2][jj] * rinvp;
              }
            p[B] = bv;
          });
          // the non-basic set itself has +1 in its null vector and weight 1: ratio 1
          const bool self = (best < 0) || !(w[B] < 1.0);
          const double alpha = self ? 1.0 : w[B];
          const int istar = self ? -1 : best;
          const int jn = kc0 + l;
          double pv[RPT];
#pragma unroll
          for (int jj = 0; jj < RPT; ++jj) {
            const int i = tid + jj * NT;
            pv[jj] = tc[l][jj];
            if (rowpt[jj] >= 0) {
              const double v = fma(alpha, pv[jj], muB[jj]);
              muB[jj] = v > 0.0 ? v : 0.0;
            }
            if (istar >= 0 && i == istar) {
              muB[jj] = 1.0 - alpha;  // the entering set keeps what is left of its unit weight
              rowpt[jj] = nbcol[jn];
            }
          }
          if (istar >= 0) {  // pivot the later own columns on row istar
#pragma unroll
            for (int l2 = l + 1; l2 < B; ++l2) {
              const double t = w[l2];
#pragma unroll
              for (int jj = 0; jj < RPT; ++jj) tc[l2][jj] = fma(-pv[jj], t, tc[l2][jj]);
            }
            if ((istar & (NT - 1)) == tid) {  // the leaving row holds the multiplier itself
              const int js = istar / NT;
#pragma unroll
              for (int jj = 0; jj < RPT; ++jj)
                if (jj == js) {
#pragma unroll
                  for (int l2 = l + 1; l2 < B; ++l2) tc[l2][jj] = w[l2];
                }
            }
#pragma unroll
            for (int jj = 0; jj < RPT; ++jj)
              if (tid + jj * NT < n) __stcg(&a.pcol[(int64_t)jn * n + tid + jj * NT], pv[jj]);
          }
          __stcg(&a.srep[(int64_t)jn * NT + tid], istar >= 0 ? istar + 2 : 1);
        }
      }
      if (k == G2 - 1) {
        if (tid == 0) stamp(a.stamps, 3);
#pragma unroll
        for (int jj = 0; jj < RPT; ++jj)
          if (rowpt[jj] >= 0 && muB[jj] > 0.0) a.omega[rowpt[jj]] = muB[jj];
      } else {
#pragma unroll
        for (int jj = 0; jj < RPT; ++jj) {
          const int i = tid + jj * NT;
          if (i < n) {
            __stcg(&a.rph[(int64_t)k * n + i], rowpt[jj] + 2);
            __stcg(&a.muh[(int64_t)k * n + i], muB[jj]);
          }
        }
      }
    }
  }
}

template <int B, int NT, int CPT, int RPT>
int launch_car2(basq_ctx* ctx, const Car2Dev& d, int grid, size_t smem) {
  BASQ_CUDA(cudaFuncSetAttribute(car2_kernel<B, NT, CPT, RPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  void* args[] = {(void*)&d};
  BASQ_CUDA(cudaLaunchCooperativeKernel((const void*)car2_kernel<B, NT, CPT, RPT>, dim3(grid), dim3(NT), args, smem,
                                        ctx->stream));
  return BASQ_OK;
}

// 512 threads: at 256 (CPT = 8, RPT = 4) the owner pivots issue fewer warp instructions, yet stage 2
// took 1.44 instead of 1.12 ms at n = 1000, S = 2000 (B200, 1000 W)
constexpr int C2_NT = 512, C2_CPT = 2048 / C2_NT, C2_RPT = 1024 / C2_NT;

}  // namespace

bool caratheodory_fast_supported(const basq_ctx* ctx, int n, int S) {
  const int m = S - n;
  return S <= C2_CPT * C2_NT && n <= C2_RPT * C2_NT && n <= 8 * ctx->num_sms && m <= 8 * ctx->num_sms && m >= 1;
}

// status_out: 0 ok, 3 = more non-basic sets than fit (A holds the stage-1 result; caller must redo)
int caratheodory_fast(basq_ctx* ctx, double* A, int n, int S, int lda, double* omega_out, int* status_out) {
  constexpr int NT = C2_NT;
  const int m_max = S;  // non-basic sets: S - rank; S - n for a full-rank system
  int B = 1;
  while (B < 8 && ((n + B - 1) / B > ctx->num_sms || (m_max + B - 1) / B > ctx->num_sms)) B *= 2;
  const int grid = std::min(ctx->num_sms, std::max((n + B - 1) / B, (m_max + B - 1) / B));
  const int G2max = grid;
  DevBuf ws;
  auto r256 = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t sz_head = 512;
  // sentinel-filled region (0xFF bytes: NaN doubles, -1 ints)
  const size_t sz_prow = r256(sizeof(double) * (size_t)n * S), sz_pcol = r256(sizeof(double) * (size_t)S * n),
               sz_prep = r256(sizeof(int) * (size_t)n * NT), sz_srep = r256(sizeof(int) * (size_t)S * NT),
               sz_muh = r256(sizeof(double) * (size_t)G2max * n), sz_rph = r256(sizeof(int) * (size_t)G2max * n);
  const size_t sz_sent = sz_prow + sz_pcol + sz_prep + sz_srep + sz_muh + sz_rph;
  const size_t sz_pinfo = r256(sizeof(int) * (size_t)n);
  BASQ_TRY(ws.alloc(ctx, sz_head + sz_sent + sz_pinfo));
  unsigned char* w = ws.as<unsigned char>();
  Car2Dev d;
  d.A = A; d.n = n; d.S = S; d.lda = lda;
  d.bar = reinterpret_cast<unsigned*>(w);            // 256 B: arrival counter + flag line
  d.status = reinterpret_cast<int*>(w + 256);
  w += sz_head;
  unsigned char* sent0 = w;
  d.prow = reinterpret_cast<double*>(w); w += sz_prow;
  d.pcol = reinterpret_cast<double*>(w); w += sz_pcol;
  d.muh = reinterpret_cast<double*>(w); w += sz_muh;
  d.prep = reinterpret_cast<int*>(w); w += sz_prep;
  d.srep = reinterpret_cast<int*>(w); w += sz_srep;
  d.rph = reinterpret_cast<int*>(w); w += sz_rph;
  d.pinfo = reinterpret_cast<int*>(w);
  d.omega = omega_out;
  d.tol = 1e-13;
  static const bool timing = [] { const char* e = getenv("BASQ_CAR_TIMING"); return e && e[0] == '1'; }();
  d.stamps = timing ? reinterpret_cast<unsigned long long*>(ws.as<unsigned char>() + 256 + 64) : nullptr;
  BASQ_CUDA(cudaMemsetAsync(ws.p, 0, sz_head, ctx->stream));
  BASQ_CUDA(cudaMemsetAsync(sent0, 0xFF, sz_sent, ctx->stream));
  const size_t smem = sizeof(int) * (size_t)S;
  switch (B) {
    case 1: BASQ_TRY((launch_car2<1, C2_NT, C2_CPT, C2_RPT>(ctx, d, grid, smem))); break;
    case 2: BASQ_TRY((launch_car2<2, C2_NT, C2_CPT, C2_RPT>(ctx, d, grid, smem))); break;
    case 4: BASQ_TRY((launch_car2<4, C2_NT, C2_CPT, C2_RPT>(ctx, d, grid, smem))); break;
    default: BASQ_TRY((launch_car2<8, C2_NT, C2_CPT, C2_RPT>(ctx, d, grid, smem))); break;
  }
  ctx->launches++;
  int status = 0;
  BASQ_CUDA(cudaMemcpyAsync(&status, d.status, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  if (timing) {
    unsigned long long t[8];
    BASQ_CUDA(cudaMemcpy(t, d.stamps, sizeof(t), cudaMemcpyDeviceToHost));
    fprintf(stderr, "[car2] n=%d S=%d B=%d grid=%d: stage1 %.1f us, barrier+list %.1f us, stage2 %.1f us; block 10: own %.2f us, hand-over to 11 %.2f us\n", n, S, B, grid,
            (t[1] - t[0]) * 1e-3, (t[2] - t[1]) * 1e-3, (t[3] - t[2]) * 1e-3, (t[5] - t[4]) * 1e-3, (t[6] - t[5]) * 1e-3);
  }
  *status_out = status;
  BASQ_CHECK(status == 0 || status == 3, BASQ_ERR_NUMERIC, "caratheodory: pivot chain watchdog fired (status %d)",
             status);
  return BASQ_OK;
}

}  // namespace basq
