// fp64 matrix product on the int8 tensor cores (Ozaki slicing, exact s32 accumulation) - see igemm.cu.
#pragma once
#include "common.cuh"

namespace basq {

constexpr int IG_DIGITS = 8;   // signed int8 digits per fp64 entry
constexpr int IG_KB = 32;      // K elements per block (the K of one int8 MMA)

// Matrix X [rows, kdim] as IG_DIGITS int8 digit matrices of the row-scaled X:
//   x[r, k] = 2^e[r] * (sum_a d_a[r, k] 2^(-7a) + residual),  |d_a| <= 64,  e[r] = (frexp exponent of max_k |x[r, k]|) - 6
// in the layout [row tile of `tile` rows][K block of 32][K half of 16][digit][tile rows][16 B]: one (row tile,
// K block) is a contiguous piece holding every digit, in the K-major no-swizzle form of the tcgen05 shared-memory
// descriptor, with consecutive digits adjacent along the rows (one MMA takes several B digits as one operand).
// The operand covers the global K positions [32 kb0, 32 (kb0 + KB)); X's column k sits at position k0 + k (dig_from_f64), positions outside X hold zero digits.
struct DigOperand {
  DevBuf dig;    // int8
  DevBuf rexp;   // int [RT * tile]: e[r]; IG_NONFINITE for a row holding Inf or NaN (its products are NaN)
  int rows = 0, tile = 0, RT = 0;
  int kb0 = 0, KB = 0;
};
constexpr int IG_NONFINITE = 1 << 30;

// op <- src (fp64, row-major, leading dimension ld) placed at global K position k0.  transposed = false: src is
// [rows, kdim]; transposed = true: src is [kdim, rows] (the operand is src^T).  tile: 128 for the left operand
// of igemm, 64 for the right one.
int dig_from_f64(basq_ctx* ctx, const double* src, int64_t ld, bool transposed, int rows, int kdim, int k0, int tile,
                 DigOperand* op);

// out[i * ldo + j] (+)= alpha * sum_k A[i, k] B[j, k] over B's K range (which A's must cover); A.tile = 128,
// B.tile = 64.  `accumulate` adds to out instead of overwriting it.
int igemm(basq_ctx* ctx, const DigOperand& A, const DigOperand& B, double alpha, double* out, int64_t ldo,
          bool accumulate);

}  // namespace basq
