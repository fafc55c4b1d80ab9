// Candidate-side stages around recombination (SURVEY 8f rows 2 and 3): candidates drawn on the
// device from the Gaussian prior, the prior's log-density, and the importance / acquisition weights
// that become `init_weights`.  All HBM-streaming elementwise kernels.
//
//   basq_sample_mvn        PriorSampler.__call__ (BASQ/_sampler.py:21-34: prior.sample),
//                          SOBER Gaussian.sample (SOBER/_prior.py:107-118)
//   basq_mvn_logpdf        prior.log_prob (BASQ/_sampler.py:136,204-212; SOBER/_prior.py:120-131)
//   basq_candidate_weights UncertaintySampler.calc_weights (BASQ/_sampler.py:190-217),
//                          PI_BQ.lfi (SOBER/_pi.py:121-139)
//   basq_cleanse_weights   WeightsStabiliser.cleansing_weights (SOBER/_weights.py:21-38)
//   basq_sir_resample      UncertaintySampler.SIR = torch.multinomial(weights, n) (BASQ/_sampler.py:104-118)
//   basq_weights_*,        the same stages on one shard of a row-sharded candidate set; the caller sums their
//   basq_sir_*             host results over the ranks (basq_b200/sharded.py)
//
// Random numbers: Philox4x32-10 (Salmon et al., SC'11), counter = (sample index lo, hi, block of 4
// dimensions, 0), key = 64-bit seed.  A sample depends only on (seed, global index), so shards drawn
// by different ranks (offset = first global row) are disjoint slices of ONE stream, whatever the
// number of ranks.  Uniforms use the top 24 bits, u = (x >> 8 + 0.5) 2^-24 in (0, 1); normals by
// Box-Muller, (x0, x1) -> (r cos 2 pi u1, r sin 2 pi u1), r = sqrt(-2 ln u0), likewise (x2, x3).
#include <math.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace basq {
namespace {

struct MvnDev {
  int d;
  double mean[BASQ_MAX_DIM];
  double chol[BASQ_MAX_DIM * (BASQ_MAX_DIM + 1) / 2];  // lower triangle, row-major packed
};

__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                       uint32_t k1, uint32_t (&out)[4]) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

template <typename T>
__global__ void sample_mvn_kernel(MvnDev p, uint64_t seed, int64_t offset, int64_t N, T* __restrict__ X) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const uint64_t g = (uint64_t)(offset + i);
  T z[BASQ_MAX_DIM];
#pragma unroll 1
  for (int blk = 0; blk * 4 < p.d; ++blk) {
    uint32_t r[4];
    philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)blk, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      // Box-Muller in fp64 for both dtypes: (k + 0.5) 2^-24 is exact there and lies strictly inside
      // (0, 1) (in fp32 half of the 24-bit draws would lose the + 0.5 to rounding and u could reach 1);
      // the fp32 stream is the rounded fp64 stream.  5e7 double log / sincospi per 1e7 x 10 candidates
      // are ~1 ms - the kernel stays bound by its N d stores.
      const double u0 = ((double)(r[2 * h] >> 8) + 0.5) * 5.9604644775390625e-08;      // 2^-24
      const double u1 = ((double)(r[2 * h + 1] >> 8) + 0.5) * 5.9604644775390625e-08;
      double sd, cd;
      sincospi(2.0 * u1, &sd, &cd);
      const double rad = sqrt(-2.0 * log(u0));
      const int k = blk * 4 + 2 * h;
      if (k < p.d) z[k] = (T)(rad * cd);
      if (k + 1 < p.d) z[k + 1] = (T)(rad * sd);
    }
  }
  // x = mean + L z
  for (int r = 0; r < p.d; ++r) {
    double acc = p.mean[r];
    const double* row = p.chol + r * (r + 1) / 2;
    for (int c = 0; c <= r; ++c) acc = fma(row[c], (double)z[c], acc);
    X[i * p.d + r] = (T)acc;
  }
}

// out[rows, cols] fp64 standard normals, the stream of sample_mvn_kernel with mean 0 / L = I and no limit
// on the number of columns: thread (row, blk) draws columns 4 blk .. 4 blk + 3.
__global__ void standard_normals_kernel(uint64_t seed, int64_t offset, int64_t rows, int cols, double* __restrict__ out) {
  const int nblk = (cols + 3) / 4;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows * nblk) return;
  const int64_t i = t / nblk;
  const int blk = (int)(t % nblk);
  const uint64_t g = (uint64_t)(offset + i);
  uint32_t r[4];
  philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)blk, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const double u0 = ((double)(r[2 * h] >> 8) + 0.5) * 5.9604644775390625e-08;      // 2^-24
    const double u1 = ((double)(r[2 * h + 1] >> 8) + 0.5) * 5.9604644775390625e-08;
    double sd, cd;
    sincospi(2.0 * u1, &sd, &cd);
    const double rad = sqrt(-2.0 * log(u0));
    const int k = blk * 4 + 2 * h;
    if (k < cols) out[i * cols + k] = rad * cd;
    if (k + 1 < cols) out[i * cols + k + 1] = rad * sd;
  }
}

// log N(x; mean, L L^T) = -1/2 |L^-1 (x - mean)|^2 - sum log L_ii - d/2 log 2 pi
template <typename T>
__global__ void mvn_logpdf_kernel(MvnDev p, double log_norm, const T* __restrict__ X, int64_t N,
                                  double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  double y[BASQ_MAX_DIM];
  double q = 0.0;
  for (int r = 0; r < p.d; ++r) {
    double acc = (double)X[i * p.d + r] - p.mean[r];
    const double* row = p.chol + r * (r + 1) / 2;
    for (int c = 0; c < r; ++c) acc = fma(-row[c], y[c], acc);
    y[r] = acc / row[r];
    q = fma(y[r], y[r], q);
  }
  out[i] = -0.5 * q + log_norm;
}

// kind 0: calc_weights, w = |m| / (ratio v + (1 - ratio) |m|)   (ratio < 1)   or |m| / (ratio v)
//         the prior density the reference multiplies into numerator and denominator cancels
//         (BASQ/_sampler.py:201-214); 0/0 -> 0 as the reference's nan never survives cleansing
// kind 1: lfi = Phi((m - 1) / sqrt(v))  (SOBER/_pi.py:132-135); log_out: log(lfi + eps32)
__global__ void candidate_weights_kernel(int kind, double ratio, int log_out, const double* __restrict__ mean,
                                         const double* __restrict__ var, int64_t N, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double m = mean[i], v = var[i];
  double w;
  if (kind == 0) {
    const double am = fabs(m);
    const double g = ratio < 1.0 ? ratio * v + (1.0 - ratio) * am : ratio * v;
    w = am / g;
    if (!(g > 0.0) && am == 0.0) w = 0.0;
  } else {
    w = normcdf((m - 1.0) / sqrt(v));
    if (log_out) w = log(w + 1.1920928955078125e-07);
  }
  out[i] = w;
}

// cleansing_weights: w < eps -> 0 ; inf / nan -> eps   (SOBER/_weights.py:32-34)
__global__ void cleanse_kernel(double* __restrict__ w, int64_t N, double eps) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  double v = w[i];
  if (v < eps) v = 0.0;
  if (isinf(v) || isnan(v)) v = eps;
  w[i] = v;
}

// deterministic sum: fixed 1024-block partials, then one block folds them in index order
__global__ void partial_sum_kernel(const double* __restrict__ w, int64_t N, double* __restrict__ part) {
  __shared__ double sh[256];
  const int64_t per = (N + gridDim.x - 1) / gridDim.x;
  const int64_t lo = (int64_t)blockIdx.x * per, hi = min(N, lo + per);
  double s = 0.0;
  for (int64_t i = lo + threadIdx.x; i < hi; i += 256) s += w[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[blockIdx.x] = sh[0];
}
__global__ void final_sum_kernel(const double* __restrict__ part, int n, double* __restrict__ total) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += part[i];
    *total = s;
  }
}
__global__ void scale_or_fill_kernel(double* __restrict__ w, int64_t N, const double* __restrict__ total) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double t = *total;
  w[i] = (t != 0.0 && isfinite(t)) ? w[i] / t : 1.0 / (double)N;
}

// ---- reproducible weight totals (basq_ctx_reproducible) ----
// max |w| (a NaN wins: its canonical bit pattern exceeds every non-negative double's); out must be zeroed
__global__ void abs_max_kernel(const double* __restrict__ w, int64_t N, unsigned long long* __restrict__ out) {
  double m = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = fabs(w[i]);
    if (!(v <= m) && m == m) m = v;
  }
  if (m != m) m = __longlong_as_double(0x7ff8000000000000ll);
  for (int o = 16; o > 0; o >>= 1) {
    const double u = __shfl_down_sync(0xffffffffu, m, o);
    if (__double_as_longlong(u) > __double_as_longlong(m)) m = u;
  }
  if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}
// hilo[0] += sum of w rounded to the grid of gm, hilo[1] += sum of the remainders on the grid of gm2: both exact,
// so the order of the atomic additions does not matter
__global__ void grid_sum_kernel(const double* __restrict__ w, int64_t N, double gm, double gm2, double* __restrict__ hilo) {
  double s = 0.0, s2 = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    const double hi = grid_round(w[i], 1.0, gm);
    s += hi;
    s2 += grid_round(w[i] - hi, 1.0, gm2);
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_down_sync(0xffffffffu, s, o);
    s2 += __shfl_down_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(hilo, s);
    atomicAdd(hilo + 1, s2);
  }
}
__global__ void add_two_kernel(const double* __restrict__ hilo, double* __restrict__ total) { *total = hilo[0] + hilo[1]; }

int weights_abs_max(basq_ctx* ctx, const double* w, int64_t N, double* max_host) {
  *max_host = 0.0;
  if (N == 0) return BASQ_OK;
  DevBuf d;
  BASQ_TRY(d.alloc(ctx, sizeof(double)));
  BASQ_CUDA(cudaMemsetAsync(d.p, 0, sizeof(double), ctx->stream));
  abs_max_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(N, 256), 4 * (int64_t)ctx->num_sms), 256, 0, ctx->stream>>>(
      w, N, d.as<unsigned long long>());
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  BASQ_CUDA(cudaMemcpyAsync(max_host, d.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

// hilo_dev[2] = the exact hi / lo sums of w[N] on the grids of N_glob weights of magnitude <= wmax (the maximum over
// every rank).  A non-finite or huge wmax makes both parts wmax: the total is not finite, as a plain sum's would be.
int weights_grid_sum(basq_ctx* ctx, const double* w, int64_t N, double wmax, int64_t N_glob, double* hilo_dev) {
  const double B = wmax * (double)N_glob;
  if (!(isfinite(B) && B < 0x1p1000)) {
    const double h[2] = {wmax == wmax ? INFINITY : wmax, 0.0};
    BASQ_CUDA(cudaMemcpyAsync(hilo_dev, h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
    return BASQ_OK;
  }
  double gm, gm2;
  grid_pair(B, (double)N_glob, &gm, &gm2);
  BASQ_CUDA(cudaMemsetAsync(hilo_dev, 0, 2 * sizeof(double), ctx->stream));
  if (N > 0) {
    grid_sum_kernel<<<(unsigned)std::min<int64_t>(ceil_div64(N, 256), 4 * (int64_t)ctx->num_sms), 256, 0, ctx->stream>>>(
        w, N, gm, gm2, hilo_dev);
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
  }
  return BASQ_OK;
}

// total_dev = the reproducible total of w[N] on one GPU: hi + lo of weights_grid_sum with the maximum of w itself
int weights_total_repro(basq_ctx* ctx, const double* w, int64_t N, double* total_dev) {
  double wmax = 0.0;
  BASQ_TRY(weights_abs_max(ctx, w, N, &wmax));
  DevBuf hilo;
  BASQ_TRY(hilo.alloc(ctx, 2 * sizeof(double)));
  BASQ_TRY(weights_grid_sum(ctx, w, N, wmax, N, hilo.as<double>()));
  add_two_kernel<<<1, 1, 0, ctx->stream>>>(hilo.as<double>(), total_dev);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));   // hilo goes out of scope
  return BASQ_OK;
}

// Sequential importance resampling without replacement (torch.multinomial(weights, n), as
// UncertaintySampler.SIR, BASQ/_sampler.py:104-118) as an exponential race (Efraimidis-Spirakis):
// key_i = -log(u_i) / w_i with u_i uniform; the n smallest keys, in increasing order, are distributed
// like n successive draws proportional to the remaining weights.  u_i = Philox(seed; i): a 53-bit
// uniform from two output words ((r0 >> 5) 2^26 + (r1 >> 6) + 0.5) 2^-53, so that the keys of 1e7+
// candidates are distinct and their gaps resolved (a 24-bit uniform has 1.6e7 values in all).
// The key of global row g with weight wi > 0; the counter depends on the row alone, so a shard that passes its
// first global row draws the same keys as the whole set.
__device__ __forceinline__ double sir_key(uint64_t g, uint64_t seed, double wi) {
  uint32_t r[4];
  philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), 0u, 0x53495200u /* "SIR" stream */, (uint32_t)seed,
                (uint32_t)(seed >> 32), r);
  const double u = ((double)(r[0] >> 5) * 67108864.0 + (double)(r[1] >> 6) + 0.5) * 1.1102230246251565e-16;  // 2^-53
  return -log(u) / wi;
}

// This kernel appends every (key, index) with key < cut to out (unordered; the host sorts the few
// survivors) and counts them.
__global__ void sir_keys_kernel(const double* __restrict__ w, int64_t N, uint64_t seed, double cut, int64_t cap,
                                double* __restrict__ key_out, int64_t* __restrict__ idx_out,
                                unsigned long long* __restrict__ count) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double wi = w[i];
  if (!(wi > 0.0)) return;
  const double key = sir_key((uint64_t)i, seed, wi);
  if (key < cut) {
    const unsigned long long slot = atomicAdd(count, 1ull);
    if ((int64_t)slot < cap) {
      key_out[slot] = key;
      idx_out[slot] = i;
    }
  }
}

// ---- the race over a sharded candidate set: device selection of the n smallest keys ------------------------
// Keys are non-negative doubles, so they order like their bit patterns as uint64.  Rows without a key (weight
// not > 0, or a key that overflowed to +inf, which basq_sir_resample never draws either) hold SIR_NO_KEY,
// which sorts after every key and falls into histogram bin SIR_BINS - 1 of the first digit (a key's sign bit
// is 0, so its first digit is below 1024).
constexpr uint64_t SIR_NO_KEY = ~0ull;
constexpr int SIR_BINS = 1 << BASQ_SIR_DIGIT_BITS;
constexpr int TILE_THREADS = 256, TILE_ITEMS = 16, TILE = TILE_THREADS * TILE_ITEMS;
constexpr unsigned FULL = 0xffffffffu;

__global__ void sir_race_keys_kernel(const double* __restrict__ w, int64_t N, uint64_t seed, int64_t idx_base,
                                     uint64_t* __restrict__ keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double wi = w[i];
  uint64_t k = SIR_NO_KEY;
  if (wi > 0.0) {
    const double key = sir_key((uint64_t)(idx_base + i), seed, wi);
    if (key < INFINITY) k = (uint64_t)__double_as_longlong(key);
  }
  keys[i] = k;
}

// hist[digit] += #{keys k : (k & mask) == bits}, digit = (k >> shift) mod SIR_BINS.  Warp-uniform loop so that
// lanes with the same digit (the leading digit holds a key's exponent: few bins, many keys) add once.
__global__ void __launch_bounds__(1024) sir_histogram_kernel(const uint64_t* __restrict__ keys, int64_t N,
                                                             uint64_t mask, uint64_t bits, int shift,
                                                             unsigned long long* __restrict__ hist) {
  __shared__ unsigned int h[SIR_BINS];
  for (int b = threadIdx.x; b < SIR_BINS; b += blockDim.x) h[b] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t b0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); b0 < N; b0 += stride) {
    const int64_t i = b0 + lane;
    unsigned dig = SIR_BINS;   // none
    if (i < N) {
      const uint64_t k = keys[i];
      if ((k & mask) == bits) dig = (unsigned)(k >> shift) & (SIR_BINS - 1);
    }
    const unsigned peers = __match_any_sync(FULL, dig);
    if (dig < SIR_BINS && lane == __ffs(peers) - 1) atomicAdd(&h[dig], (unsigned)__popc(peers));
  }
  __syncthreads();
  for (int b = threadIdx.x; b < SIR_BINS; b += blockDim.x)
    if (h[b]) atomicAdd(&hist[b], (unsigned long long)h[b]);
}

// Exclusive prefix sum of a[n] in place (one block of 1024 threads, each folding a contiguous run), total out.
__global__ void __launch_bounds__(1024) exclusive_scan_kernel(int64_t* __restrict__ a, int64_t n,
                                                              int64_t* __restrict__ total) {
  __shared__ int64_t part[1024];
  const int t = threadIdx.x;
  const int64_t per = (n + 1023) / 1024, lo = min(n, t * per), hi = min(n, lo + per);
  int64_t s = 0;
  for (int64_t i = lo; i < hi; ++i) s += a[i];
  part[t] = s;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int64_t v = t >= o ? part[t - o] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  s = part[t] - s;
  for (int64_t i = lo; i < hi; ++i) {
    const int64_t v = a[i];
    a[i] = s;
    s += v;
  }
  if (t == 1023 && total) *total = part[1023];
}

// Exclusive scan of one flag per thread across a block of TILE_THREADS; returns the block's total.
__device__ __forceinline__ int block_scan_flag(bool f, int* rank, int* warp_tot /* smem [8] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned bal = __ballot_sync(FULL, f);
  if (lane == 0) warp_tot[warp] = __popc(bal);
  __syncthreads();
  int before = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < TILE_THREADS / 32; ++w) {
    before += w < warp ? warp_tot[w] : 0;
    tot += warp_tot[w];
  }
  __syncthreads();
  *rank = before + __popc(bal & ((1u << lane) - 1u));
  return tot;
}

// Collect: tile counts of keys <= T, then an order-preserving write of (key, global index) at the scanned offsets.
__global__ void __launch_bounds__(TILE_THREADS) sir_tile_count_kernel(const uint64_t* __restrict__ keys, int64_t N,
                                                                      uint64_t T, int64_t* __restrict__ counts) {
  __shared__ int warp_tot[TILE_THREADS / 32];
  const int64_t t0 = (int64_t)blockIdx.x * TILE;
  int c = 0;
#pragma unroll 4
  for (int r = 0; r < TILE_ITEMS; ++r) {
    const int64_t i = t0 + r * TILE_THREADS + threadIdx.x;
    c += (i < N && keys[i] <= T) ? 1 : 0;
  }
  c = __reduce_add_sync(FULL, c);
  if ((threadIdx.x & 31) == 0) warp_tot[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < TILE_THREADS / 32; ++w) s += warp_tot[w];
    counts[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(TILE_THREADS) sir_collect_kernel(const uint64_t* __restrict__ keys, int64_t N,
                                                                   uint64_t T, int64_t idx_base,
                                                                   const int64_t* __restrict__ offsets,
                                                                   uint64_t* __restrict__ keys_out,
                                                                   int64_t* __restrict__ idx_out) {
  __shared__ int warp_tot[TILE_THREADS / 32];
  const int64_t t0 = (int64_t)blockIdx.x * TILE;
  int64_t pos = offsets[blockIdx.x];
  for (int r = 0; r < TILE_ITEMS; ++r) {
    const int64_t i = t0 + r * TILE_THREADS + threadIdx.x;
    const uint64_t k = i < N ? keys[i] : SIR_NO_KEY;
    const bool take = i < N && k <= T;
    int rank;
    const int tot = block_scan_flag(take, &rank, warp_tot);
    if (take) {
      keys_out[pos + rank] = k;
      idx_out[pos + rank] = idx_base + i;
    }
    pos += tot;
  }
}

// Stable LSD radix sort of (key, index) pairs, 8-bit digits: per-tile digit counts (digit-major, so that one
// exclusive scan gives every tile its output offset per digit), then a scatter that ranks each round of
// TILE_THREADS pairs by (warp, lane) within its digit - the input order is kept among equal digits.
constexpr int SORT_BINS = 256;

__global__ void __launch_bounds__(TILE_THREADS) sort_tile_hist_kernel(const uint64_t* __restrict__ keys, int64_t K,
                                                                      int shift, int64_t nb,
                                                                      int64_t* __restrict__ counts) {
  __shared__ int h[SORT_BINS];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int64_t t0 = (int64_t)blockIdx.x * TILE;
#pragma unroll 4
  for (int r = 0; r < TILE_ITEMS; ++r) {
    const int64_t i = t0 + r * TILE_THREADS + threadIdx.x;
    if (i < K) atomicAdd(&h[(unsigned)(keys[i] >> shift) & (SORT_BINS - 1)], 1);
  }
  __syncthreads();
  counts[(int64_t)threadIdx.x * nb + blockIdx.x] = h[threadIdx.x];
}

__global__ void __launch_bounds__(TILE_THREADS) sort_scatter_kernel(const uint64_t* __restrict__ keys_in,
                                                                    const int64_t* __restrict__ idx_in, int64_t K,
                                                                    int shift, int64_t nb,
                                                                    const int64_t* __restrict__ offsets,
                                                                    uint64_t* __restrict__ keys_out,
                                                                    int64_t* __restrict__ idx_out) {
  constexpr int WARPS = TILE_THREADS / 32;
  __shared__ int64_t base[SORT_BINS];
  __shared__ int warp_cnt[WARPS][SORT_BINS];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  base[t] = offsets[(int64_t)t * nb + blockIdx.x];
#pragma unroll
  for (int w = 0; w < WARPS; ++w) warp_cnt[w][t] = 0;
  __syncthreads();
  const int64_t t0 = (int64_t)blockIdx.x * TILE;
  for (int r = 0; r < TILE_ITEMS; ++r) {
    const int64_t i = t0 + r * TILE_THREADS + t;
    if (t0 + r * TILE_THREADS >= K) break;              // block-uniform
    const bool valid = i < K;
    const uint64_t k = valid ? keys_in[i] : 0;
    const unsigned dig = valid ? (unsigned)(k >> shift) & (SORT_BINS - 1) : SORT_BINS;
    const unsigned peers = __match_any_sync(FULL, dig);
    const int lt = __popc(peers & ((1u << lane) - 1u));
    if (valid && lt == 0) warp_cnt[warp][dig] = __popc(peers);
    __syncthreads();
    if (valid) {
      int64_t p = base[dig] + lt;
      for (int w = 0; w < warp; ++w) p += warp_cnt[w][dig];
      keys_out[p] = k;
      idx_out[p] = idx_in[i];
    }
    __syncthreads();
    int64_t add = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) {
      add += warp_cnt[w][t];
      warp_cnt[w][t] = 0;
    }
    base[t] += add;
    __syncthreads();
  }
}

__global__ void normalise_kernel(double* __restrict__ w, int64_t N, double total, double fill) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  w[i] = (total != 0.0 && isfinite(total)) ? w[i] / total : fill;
}

int pack_mvn(int d, const double* mean_host, const double* chol_host, MvnDev* p, double* log_norm) {
  BASQ_CHECK(d >= 1 && d <= BASQ_MAX_DIM, BASQ_ERR_INVALID, "mvn: dimension %d out of range", d);
  BASQ_CHECK(mean_host && chol_host, BASQ_ERR_INVALID, "mvn: NULL parameter");
  p->d = d;
  double ld = 0.0;
  for (int r = 0; r < d; ++r) {
    p->mean[r] = mean_host[r];
    for (int c = 0; c <= r; ++c) p->chol[r * (r + 1) / 2 + c] = chol_host[r * d + c];
    BASQ_CHECK(chol_host[r * d + r] > 0.0, BASQ_ERR_INVALID, "mvn: Cholesky factor has a non-positive diagonal");
    ld += log(chol_host[r * d + r]);
  }
  if (log_norm) *log_norm = -ld - 0.5 * d * 1.8378770664093453;  // log(2 pi)
  return BASQ_OK;
}

}  // namespace

int sum_device(basq_ctx* ctx, const double* w, int64_t N, double* total_dev) {
  constexpr int NB = 1024;
  DevBuf part;
  BASQ_TRY(part.alloc(ctx, sizeof(double) * NB));
  partial_sum_kernel<<<NB, 256, 0, ctx->stream>>>(w, N, part.as<double>());
  final_sum_kernel<<<1, 32, 0, ctx->stream>>>(part.as<double>(), NB, total_dev);
  ctx->launches += 2;
  BASQ_CUDA(cudaGetLastError());
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));  // part goes out of scope
  return BASQ_OK;
}

int standard_normals(basq_ctx* ctx, uint64_t seed, int64_t offset, int64_t rows, int cols, double* out) {
  if (rows == 0 || cols == 0) return BASQ_OK;
  const int64_t threads = rows * ((cols + 3) / 4);
  standard_normals_kernel<<<(unsigned)ceil_div64(threads, 256), 256, 0, ctx->stream>>>(seed, offset, rows, cols, out);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

}  // namespace basq

using namespace basq;


extern "C" {

int basq_standard_normals(basq_ctx* ctx, uint64_t seed, int64_t offset, int64_t rows, int cols, double* out) {
  BASQ_CHECK(ctx && (out || rows == 0 || cols == 0), BASQ_ERR_INVALID, "basq_standard_normals: NULL argument");
  BASQ_CHECK(rows >= 0 && cols >= 0 && offset >= 0, BASQ_ERR_INVALID, "basq_standard_normals: negative size or offset");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  return standard_normals(ctx, seed, offset, rows, cols, out);
}

int basq_sample_mvn(basq_ctx* ctx, uint64_t seed, int64_t offset, int64_t N, int d, int dtype,
                    const double* mean_host, const double* chol_host, void* X_out) {
  BASQ_CHECK(ctx && (X_out || N == 0), BASQ_ERR_INVALID, "basq_sample_mvn: NULL argument");
  BASQ_CHECK(N >= 0 && offset >= 0, BASQ_ERR_INVALID, "basq_sample_mvn: negative size or offset");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  MvnDev p;
  BASQ_TRY(pack_mvn(d, mean_host, chol_host, &p, nullptr));
  if (N == 0) return BASQ_OK;
  const unsigned blocks = (unsigned)ceil_div64(N, 256);
  if (dtype == BASQ_F32) sample_mvn_kernel<float><<<blocks, 256, 0, ctx->stream>>>(p, seed, offset, N, (float*)X_out);
  else sample_mvn_kernel<double><<<blocks, 256, 0, ctx->stream>>>(p, seed, offset, N, (double*)X_out);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

int basq_mvn_logpdf(basq_ctx* ctx, const void* X, int64_t N, int d, int dtype, const double* mean_host,
                    const double* chol_host, double* out) {
  BASQ_CHECK(ctx && (X || N == 0) && out, BASQ_ERR_INVALID, "basq_mvn_logpdf: NULL argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  MvnDev p;
  double log_norm = 0.0;
  BASQ_TRY(pack_mvn(d, mean_host, chol_host, &p, &log_norm));
  if (N == 0) return BASQ_OK;
  const unsigned blocks = (unsigned)ceil_div64(N, 256);
  if (dtype == BASQ_F32) mvn_logpdf_kernel<float><<<blocks, 256, 0, ctx->stream>>>(p, log_norm, (const float*)X, N, out);
  else mvn_logpdf_kernel<double><<<blocks, 256, 0, ctx->stream>>>(p, log_norm, (const double*)X, N, out);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

int basq_candidate_weights(basq_ctx* ctx, int kind, double ratio, int log_out, const double* mean, const double* var,
                           int64_t N, int normalise, double* w_out) {
  BASQ_CHECK(ctx && mean && var && w_out, BASQ_ERR_INVALID, "basq_candidate_weights: NULL argument");
  BASQ_CHECK(kind == 0 || kind == 1, BASQ_ERR_INVALID, "basq_candidate_weights: unknown kind %d", kind);
  BASQ_CHECK(kind != 0 || (ratio >= 0.0 && ratio <= 1.0), BASQ_ERR_INVALID, "calc_weights: ratio must lie in [0, 1]");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  if (N <= 0) return BASQ_OK;
  const unsigned blocks = (unsigned)ceil_div64(N, 256);
  candidate_weights_kernel<<<blocks, 256, 0, ctx->stream>>>(kind, ratio, log_out, mean, var, N, w_out);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  if (normalise) {
    DevBuf total;
    BASQ_TRY(total.alloc(ctx, sizeof(double)));
    if (ctx->reproducible) BASQ_TRY(weights_total_repro(ctx, w_out, N, total.as<double>()));
    else BASQ_TRY(sum_device(ctx, w_out, N, total.as<double>()));
    scale_or_fill_kernel<<<blocks, 256, 0, ctx->stream>>>(w_out, N, total.as<double>());
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return BASQ_OK;
}

int basq_sir_resample(basq_ctx* ctx, const double* w, int64_t N, int64_t n_out, uint64_t seed, int64_t* idx_out_host,
                      int64_t* n_drawn_host) {
  BASQ_CHECK(ctx && w && idx_out_host && n_drawn_host, BASQ_ERR_INVALID, "basq_sir_resample: NULL argument");
  BASQ_CHECK(N >= 1 && n_out >= 0, BASQ_ERR_INVALID, "basq_sir_resample: bad sizes");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  *n_drawn_host = 0;
  if (n_out == 0) return BASQ_OK;
  DevBuf total, keys, idxs, count;
  BASQ_TRY(total.alloc(ctx, sizeof(double)));
  BASQ_TRY(sum_device(ctx, w, N, total.as<double>()));
  double tot = 0.0;
  BASQ_CUDA(cudaMemcpyAsync(&tot, total.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  BASQ_CHECK(isfinite(tot) && tot > 0.0, BASQ_ERR_NUMERIC, "basq_sir_resample: weights sum to %g", tot);
  const int64_t want = std::min<int64_t>(n_out, N);
  const int64_t cap = std::min<int64_t>(N, 4 * want + 4096);
  BASQ_TRY(keys.alloc(ctx, sizeof(double) * cap));
  BASQ_TRY(idxs.alloc(ctx, sizeof(int64_t) * cap));
  BASQ_TRY(count.alloc(ctx, sizeof(unsigned long long)));
  // #keys below t is about t * sum(w) while t * max(w) << 1: start 50 % above the target, double on a miss
  double cut = 1.5 * (double)want / tot + 1e-300;
  unsigned long long got = 0;
  for (int attempt = 0; attempt < 80; ++attempt) {
    BASQ_CUDA(cudaMemsetAsync(count.p, 0, sizeof(unsigned long long), ctx->stream));
    sir_keys_kernel<<<(unsigned)ceil_div64(N, 256), 256, 0, ctx->stream>>>(w, N, seed, cut, cap, keys.as<double>(),
                                                                           idxs.as<int64_t>(),
                                                                           count.as<unsigned long long>());
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
    BASQ_CUDA(cudaMemcpyAsync(&got, count.p, sizeof(got), cudaMemcpyDeviceToHost, ctx->stream));
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
    if ((int64_t)got > cap) { cut *= 0.6; continue; }            // overshoot: more survivors than the buffer holds
    if ((int64_t)got >= want || !isfinite(cut)) break;            // enough (or every positive weight is in)
    cut = (cut > 1e300) ? INFINITY : cut * 2.0;
  }
  BASQ_CHECK((int64_t)got <= cap, BASQ_ERR_NUMERIC, "basq_sir_resample: could not bracket the %lld-th key", (long long)want);
  std::vector<double> hk((size_t)got);
  std::vector<int64_t> hi((size_t)got);
  BASQ_CUDA(cudaMemcpyAsync(hk.data(), keys.p, sizeof(double) * got, cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaMemcpyAsync(hi.data(), idxs.p, sizeof(int64_t) * got, cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  std::vector<int64_t> order((size_t)got);
  for (size_t t = 0; t < order.size(); ++t) order[t] = (int64_t)t;
  std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
    return hk[a] < hk[b] || (hk[a] == hk[b] && hi[a] < hi[b]);
  });
  const int64_t take = std::min<int64_t>(want, (int64_t)got);   // fewer than n positive weights: all of them
  for (int64_t t = 0; t < take; ++t) idx_out_host[t] = hi[order[t]];
  *n_drawn_host = take;
  return BASQ_OK;
}

int basq_cleanse_weights(basq_ctx* ctx, double* w, int64_t N, double eps) {
  BASQ_CHECK(ctx && (w || N == 0), BASQ_ERR_INVALID, "basq_cleanse_weights: NULL argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  if (N <= 0) return BASQ_OK;
  const unsigned blocks = (unsigned)ceil_div64(N, 256);
  cleanse_kernel<<<blocks, 256, 0, ctx->stream>>>(w, N, eps);
  ctx->launches++;
  DevBuf total;
  BASQ_TRY(total.alloc(ctx, sizeof(double)));
  if (ctx->reproducible) BASQ_TRY(weights_total_repro(ctx, w, N, total.as<double>()));
  else BASQ_TRY(sum_device(ctx, w, N, total.as<double>()));
  scale_or_fill_kernel<<<blocks, 256, 0, ctx->stream>>>(w, N, total.as<double>());
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

int basq_weights_sum(basq_ctx* ctx, const double* w, int64_t N, double* total_host) {
  BASQ_CHECK(ctx && (w || N == 0) && total_host, BASQ_ERR_INVALID, "basq_weights_sum: NULL argument");
  BASQ_CHECK(N >= 0, BASQ_ERR_INVALID, "basq_weights_sum: negative size");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  *total_host = 0.0;
  if (N == 0) return BASQ_OK;
  DevBuf total;
  BASQ_TRY(total.alloc(ctx, sizeof(double)));
  BASQ_TRY(sum_device(ctx, w, N, total.as<double>()));
  BASQ_CUDA(cudaMemcpyAsync(total_host, total.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

int basq_weights_max(basq_ctx* ctx, const double* w, int64_t N, double* max_host) {
  BASQ_CHECK(ctx && (w || N == 0) && max_host && N >= 0, BASQ_ERR_INVALID, "basq_weights_max: bad argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  return weights_abs_max(ctx, w, N, max_host);
}

int basq_weights_sum_grid(basq_ctx* ctx, const double* w, int64_t N, double wmax, int64_t N_glob, double* hilo_host) {
  BASQ_CHECK(ctx && (w || N == 0) && hilo_host && N >= 0 && N_glob >= N && N_glob >= 1, BASQ_ERR_INVALID,
             "basq_weights_sum_grid: bad argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  DevBuf hilo;
  BASQ_TRY(hilo.alloc(ctx, 2 * sizeof(double)));
  BASQ_TRY(weights_grid_sum(ctx, w, N, wmax, N_glob, hilo.as<double>()));
  BASQ_CUDA(cudaMemcpyAsync(hilo_host, hilo.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

int basq_weights_normalise(basq_ctx* ctx, double* w, int64_t N_loc, double total, int64_t N_glob) {
  BASQ_CHECK(ctx && (w || N_loc == 0), BASQ_ERR_INVALID, "basq_weights_normalise: NULL argument");
  BASQ_CHECK(N_loc >= 0 && N_glob >= N_loc && N_glob >= 1, BASQ_ERR_INVALID,
             "basq_weights_normalise: bad sizes (N_loc %lld, N_glob %lld)", (long long)N_loc, (long long)N_glob);
  BASQ_CUDA(cudaSetDevice(ctx->device));
  if (N_loc == 0) return BASQ_OK;
  normalise_kernel<<<(unsigned)ceil_div64(N_loc, 256), 256, 0, ctx->stream>>>(w, N_loc, total, 1.0 / (double)N_glob);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

int basq_weights_cleanse(basq_ctx* ctx, double* w, int64_t N, double eps) {
  BASQ_CHECK(ctx && (w || N == 0), BASQ_ERR_INVALID, "basq_weights_cleanse: NULL argument");
  BASQ_CHECK(N >= 0, BASQ_ERR_INVALID, "basq_weights_cleanse: negative size");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  if (N == 0) return BASQ_OK;
  cleanse_kernel<<<(unsigned)ceil_div64(N, 256), 256, 0, ctx->stream>>>(w, N, eps);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

int basq_sir_keys(basq_ctx* ctx, const double* w, int64_t N_loc, uint64_t seed, int64_t idx_base, uint64_t* keys_out) {
  BASQ_CHECK(ctx && ((w && keys_out) || N_loc == 0), BASQ_ERR_INVALID, "basq_sir_keys: NULL argument");
  BASQ_CHECK(N_loc >= 0 && idx_base >= 0, BASQ_ERR_INVALID, "basq_sir_keys: negative size or index base");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  if (N_loc == 0) return BASQ_OK;
  sir_race_keys_kernel<<<(unsigned)ceil_div64(N_loc, 256), 256, 0, ctx->stream>>>(w, N_loc, seed, idx_base, keys_out);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

int basq_sir_histogram(basq_ctx* ctx, const uint64_t* keys, int64_t N_loc, uint64_t mask, uint64_t bits, int shift,
                       int64_t* hist_host) {
  BASQ_CHECK(ctx && (keys || N_loc == 0) && hist_host, BASQ_ERR_INVALID, "basq_sir_histogram: NULL argument");
  BASQ_CHECK(N_loc >= 0 && shift >= 0 && shift < 64, BASQ_ERR_INVALID, "basq_sir_histogram: bad size or shift");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  for (int b = 0; b < SIR_BINS; ++b) hist_host[b] = 0;
  if (N_loc == 0) return BASQ_OK;
  DevBuf hist;
  BASQ_TRY(hist.alloc(ctx, sizeof(unsigned long long) * SIR_BINS));
  BASQ_CUDA(cudaMemsetAsync(hist.p, 0, sizeof(unsigned long long) * SIR_BINS, ctx->stream));
  const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div64(N_loc, 1024), 2 * std::max(ctx->num_sms, 1));
  sir_histogram_kernel<<<blocks, 1024, 0, ctx->stream>>>(keys, N_loc, mask, bits, shift,
                                                          hist.as<unsigned long long>());
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  BASQ_CUDA(cudaMemcpyAsync(hist_host, hist.p, sizeof(int64_t) * SIR_BINS, cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

int basq_sir_collect(basq_ctx* ctx, const uint64_t* keys, int64_t N_loc, uint64_t T, int64_t idx_base, int64_t cap,
                     uint64_t* keys_out, int64_t* idx_out, int64_t* n_out_host) {
  BASQ_CHECK(ctx && (keys || N_loc == 0) && ((keys_out && idx_out) || cap == 0) && n_out_host, BASQ_ERR_INVALID,
             "basq_sir_collect: NULL argument");
  BASQ_CHECK(N_loc >= 0 && cap >= 0 && idx_base >= 0, BASQ_ERR_INVALID, "basq_sir_collect: negative argument");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  *n_out_host = 0;
  if (N_loc == 0) return BASQ_OK;
  const int64_t nb = ceil_div64(N_loc, TILE);
  DevBuf offs, total;
  BASQ_TRY(offs.alloc(ctx, sizeof(int64_t) * nb));
  BASQ_TRY(total.alloc(ctx, sizeof(int64_t)));
  sir_tile_count_kernel<<<(unsigned)nb, TILE_THREADS, 0, ctx->stream>>>(keys, N_loc, T, offs.as<int64_t>());
  exclusive_scan_kernel<<<1, 1024, 0, ctx->stream>>>(offs.as<int64_t>(), nb, total.as<int64_t>());
  ctx->launches += 2;
  BASQ_CUDA(cudaGetLastError());
  int64_t n = 0;
  BASQ_CUDA(cudaMemcpyAsync(&n, total.p, sizeof(n), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  BASQ_CHECK(n <= cap, BASQ_ERR_INVALID, "basq_sir_collect: %lld keys <= T, room for %lld", (long long)n,
             (long long)cap);
  *n_out_host = n;
  if (n == 0) return BASQ_OK;
  sir_collect_kernel<<<(unsigned)nb, TILE_THREADS, 0, ctx->stream>>>(keys, N_loc, T, idx_base, offs.as<int64_t>(),
                                                                     keys_out, idx_out);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

int basq_sir_sort(basq_ctx* ctx, uint64_t* keys, int64_t* idx, int64_t K) {
  BASQ_CHECK(ctx && ((keys && idx) || K == 0), BASQ_ERR_INVALID, "basq_sir_sort: NULL argument");
  BASQ_CHECK(K >= 0, BASQ_ERR_INVALID, "basq_sir_sort: negative size");
  BASQ_CUDA(cudaSetDevice(ctx->device));
  if (K <= 1) return BASQ_OK;
  const int64_t nb = ceil_div64(K, TILE);
  DevBuf kt, it, counts;
  BASQ_TRY(kt.alloc(ctx, sizeof(uint64_t) * K));
  BASQ_TRY(it.alloc(ctx, sizeof(int64_t) * K));
  BASQ_TRY(counts.alloc(ctx, sizeof(int64_t) * SORT_BINS * nb));
  uint64_t* kb[2] = {keys, kt.as<uint64_t>()};
  int64_t* ib[2] = {idx, it.as<int64_t>()};
  for (int pass = 0; pass < 8; ++pass) {      // even number of passes: the result lands back in keys / idx
    const int src = pass & 1, shift = 8 * pass;
    sort_tile_hist_kernel<<<(unsigned)nb, TILE_THREADS, 0, ctx->stream>>>(kb[src], K, shift, nb, counts.as<int64_t>());
    exclusive_scan_kernel<<<1, 1024, 0, ctx->stream>>>(counts.as<int64_t>(), SORT_BINS * nb, nullptr);
    sort_scatter_kernel<<<(unsigned)nb, TILE_THREADS, 0, ctx->stream>>>(kb[src], ib[src], K, shift, nb,
                                                                        counts.as<int64_t>(), kb[1 - src], ib[1 - src]);
    ctx->launches += 3;
    BASQ_CUDA(cudaGetLastError());
  }
  return BASQ_OK;
}

}  // extern "C"
