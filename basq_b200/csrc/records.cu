// Candidate records: build (with zero-weight filtering), per-set masses, per-round reweight +
// order-preserving compaction, result extraction.  All HBM-streaming kernels.
#include "common.cuh"
#include "prep.cuh"

namespace basq {

// ---------------------------------------------------------------------------------------------
// build
// ---------------------------------------------------------------------------------------------
// pass 1: number of kept (mu != 0) points per 256-point block
__global__ void count_kept_kernel(const double* __restrict__ mu, int64_t N, int* __restrict__ counts) {
  const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const bool keep = (p < N) && (mu[p] != 0.0);
  const int c = __syncthreads_count(keep);
  if (threadIdx.x == 0) counts[blockIdx.x] = c;
}

// pass 2: exclusive scan of the block counts (single block, chunked; deterministic)
__global__ void scan_counts_kernel(const int* __restrict__ counts, int nb, int64_t* __restrict__ offsets,
                                   int64_t* __restrict__ total) {
  __shared__ int64_t sh[1024];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < nb; base += 1024) {
    const int i = base + threadIdx.x;
    const int64_t v = (i < nb) ? counts[i] : 0;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
      int64_t t = 0;
      if ((int)threadIdx.x >= off) t = sh[threadIdx.x - off];
      __syncthreads();
      sh[threadIdx.x] += t;
      __syncthreads();
    }
    if (i < nb) offsets[i] = carry + sh[threadIdx.x] - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry += sh[1023];
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

template <typename T>
__device__ __forceinline__ void write_record_f32(const KParams& kp, unsigned char* rec, int rec_bytes, const T* x,
                                                 double wf, double mu, int idx) {
  float xs[BASQ_MAX_DIM];
  float nrm;
  prep_point_f32(kp, x, xs, &nrm);
  double* h = reinterpret_cast<double*>(rec);
  h[0] = wf;
  h[1] = mu;
  reinterpret_cast<int*>(rec)[4] = idx;
  float* f = reinterpret_cast<float*>(rec);
  f[5] = point_a_term(kp, nrm);
  const int nf = rec_bytes / 4;
  for (int i = 6; i < nf; ++i) f[i] = (i - 6 < kp.dp) ? xs[i - 6] : 0.f;
}

template <typename T>
__device__ __forceinline__ void write_record_f64(const KParams& kp, unsigned char* rec, int rec_bytes, const T* x,
                                                 double wf, double mu, int64_t idx) {
  double xs[BASQ_MAX_DIM];
  prep_point_f64(kp, x, xs);
  double* h = reinterpret_cast<double*>(rec);
  h[0] = wf;
  h[1] = mu;
  reinterpret_cast<int64_t*>(rec)[2] = idx;
  const int nd = rec_bytes / 8;
  for (int i = 3; i < nd; ++i) h[i] = (i - 3 < kp.dp) ? xs[i - 3] : 0.0;
}

// pass 3 (or the only pass when mu == nullptr): write the records of the kept points in order.
// The kept records of a block are contiguous in the pool (slot = rank of the point among the block's
// kept points), so they are assembled in shared memory and streamed out with 16-byte stores that
// consecutive threads issue to consecutive addresses.
template <typename T, bool F64>
__global__ void build_records_kernel(KParams kp, const T* __restrict__ X, int64_t N, double uniform_w,
                                     const double* __restrict__ mu, const double* __restrict__ factor,
                                     int factor_in_weight, const int64_t* __restrict__ block_off,
                                     unsigned char* __restrict__ recs, int rec_bytes) {
  extern __shared__ __align__(16) unsigned char stage_rec[];  // [256][rec_bytes]
  __shared__ int warp_tot[8];
  const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const double m = (p < N) ? (mu ? mu[p] : uniform_w) : 0.0;
  const bool keep = (p < N) && (m != 0.0);
  const unsigned bal = __ballot_sync(0xffffffffu, keep);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int pre = __popc(bal & ((1u << lane) - 1u));
  if (lane == 0) warp_tot[warp] = __popc(bal);
  __syncthreads();
  int wbase = 0, kept = 0;
  for (int w = 0; w < 8; ++w) {
    if (w < warp) wbase += warp_tot[w];
    kept += warp_tot[w];
  }
  if (keep) {
    const double fac = factor ? factor[p] : 1.0;
    const double wf = factor_in_weight ? m * fac : fac;
    unsigned char* rec = stage_rec + (size_t)(wbase + pre) * rec_bytes;
    if (F64)
      write_record_f64(kp, rec, rec_bytes, X + p * kp.d, wf, m, p);
    else
      write_record_f32(kp, rec, rec_bytes, X + p * kp.d, wf, m, (int)p);
  }
  __syncthreads();
  const int64_t first = mu ? block_off[blockIdx.x] : (int64_t)blockIdx.x * 256;
  uint4* dst = reinterpret_cast<uint4*>(recs + first * (int64_t)rec_bytes);
  const uint4* src = reinterpret_cast<const uint4*>(stage_rec);
  const int chunks = kept * (rec_bytes / 16);
  for (int c = threadIdx.x; c < chunks; c += 256) dst[c] = src[c];
}

int build_records(basq_ctx* ctx, const KParams& kp, int dtype, const void* X, int64_t N, double uniform_w,
                  const double* mu, const double* factor, bool factor_in_weight, RecPool* pool, bool round_buffer) {
  BASQ_CHECK(N >= 0 && N < (1ll << 31) - 1024, BASQ_ERR_UNSUPPORTED,
             "at most 2^31 candidates per rank (got %lld)", (long long)N);
  pool->dtype = dtype;
  pool->dp = kp.dp;
  pool->rec_bytes = (dtype == BASQ_F32) ? rec_bytes_f32(kp.dp) : rec_bytes_f64(kp.dp);
  pool->cur = 0;
  pool->count = 0;
  pool->capacity = N;
  BASQ_TRY(pool->buf[0].alloc(ctx, (size_t)(N + 1) * pool->rec_bytes));
  // the second buffer only ever receives the survivors of a round (about half), but the first
  // round of a weighted run may keep more: size it for the worst case of one halving round + 1.
  if (round_buffer) BASQ_TRY(pool->buf[1].alloc(ctx, (size_t)(N + 1) * pool->rec_bytes));
  if (N == 0) return BASQ_OK;
  const int nb = ceil_div(N, 256);
  DevBuf counts, offs, total;
  int64_t kept = N;
  if (mu) {
    BASQ_TRY(counts.alloc(ctx, sizeof(int) * nb));
    BASQ_TRY(offs.alloc(ctx, sizeof(int64_t) * nb));
    BASQ_TRY(total.alloc(ctx, sizeof(int64_t)));
    count_kept_kernel<<<nb, 256, 0, ctx->stream>>>(mu, N, counts.as<int>());
    scan_counts_kernel<<<1, 1024, 0, ctx->stream>>>(counts.as<int>(), nb, offs.as<int64_t>(), total.as<int64_t>());
    ctx->launches += 2;
  }
  unsigned char* recs = pool->buf[0].as<unsigned char>();
  const int64_t* boff = mu ? offs.as<int64_t>() : nullptr;
  const size_t smem = (size_t)256 * pool->rec_bytes;
  if (dtype == BASQ_F32) {
    BASQ_CUDA(cudaFuncSetAttribute(build_records_kernel<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    build_records_kernel<float, false><<<nb, 256, smem, ctx->stream>>>(kp, (const float*)X, N, uniform_w, mu, factor,
                                                                     factor_in_weight ? 1 : 0, boff, recs,
                                                                     pool->rec_bytes);
  } else {
    BASQ_CUDA(cudaFuncSetAttribute(build_records_kernel<double, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    build_records_kernel<double, true><<<nb, 256, smem, ctx->stream>>>(kp, (const double*)X, N, uniform_w, mu, factor,
                                                                      factor_in_weight ? 1 : 0, boff, recs,
                                                                      pool->rec_bytes);
  }
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  if (mu) {
    BASQ_CUDA(cudaMemcpyAsync(&kept, total.p, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  pool->count = kept;
  return BASQ_OK;
}

// ---------------------------------------------------------------------------------------------
// set masses: mass[j] = sum of mu over local points whose global position = j (mod S)
// ---------------------------------------------------------------------------------------------
// REPRO: every mass is rounded to the grid of gm before it is added (grid_round, common.cuh), its remainder to the
// finer grid of gm2 and summed into mass2
template <bool REPRO>
__global__ void set_mass_kernel(const unsigned char* __restrict__ recs, int rec_bytes, int64_t count, int64_t off,
                                int S, int S_eff, double* __restrict__ mass, double gm, double gm2,
                                double* __restrict__ mass2) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= S) return;
  double s = 0.0, s2 = 0.0;
  if (warp < S_eff) {
    int64_t p0 = ((int64_t)warp - off) % S;
    if (p0 < 0) p0 += S;
    for (int64_t p = p0 + (int64_t)lane * S; p < count; p += (int64_t)32 * S) {
      const double m = reinterpret_cast<const double*>(recs + p * rec_bytes)[1];
      if (REPRO) {
        const double hi = grid_round(m, 1.0, gm);
        s += hi;
        s2 += grid_round(m - hi, 1.0, gm2);
      } else {
        s += m;
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (REPRO)
    for (int o = 16; o > 0; o >>= 1) s2 += __shfl_down_sync(0xffffffffu, s2, o);
  if (lane == 0) mass[warp] = s;
  if (REPRO && lane == 0) mass2[warp] = s2;
}

int set_masses(basq_ctx* ctx, const RecPool& pool, int64_t off_glob, int S, int S_eff, double* mass_out, double grid_m,
               double grid_m2, double* mass_out2) {
  const int threads = 256;
  const int blocks = ceil_div((int64_t)S * 32, threads);
  if (grid_m != 0.0)
    set_mass_kernel<true><<<blocks, threads, 0, ctx->stream>>>(pool.buf[pool.cur].as<unsigned char>(), pool.rec_bytes,
                                                               pool.count, off_glob, S, S_eff, mass_out, grid_m,
                                                               grid_m2, mass_out2);
  else
    set_mass_kernel<false><<<blocks, threads, 0, ctx->stream>>>(pool.buf[pool.cur].as<unsigned char>(), pool.rec_bytes,
                                                                pool.count, off_glob, S, S_eff, mass_out, 0.0, 0.0,
                                                                nullptr);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

// cell objective sums: out[j] = sum of mu_p * obj[idx_p] over local points in cell j (the extra row
// of the objective-aware recombination, SOBER/_rchq.py:138-146); obj is indexed by the candidate's
// original local row, which every record carries
template <bool REPRO>
__global__ void cell_obj_kernel(const unsigned char* __restrict__ recs, int rec_bytes, int f64, int64_t count,
                                int64_t off, int S, int S_eff, const double* __restrict__ obj,
                                double* __restrict__ out, double gm, double gm2, double* __restrict__ out2) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= S) return;
  double s = 0.0, s2 = 0.0;
  if (warp < S_eff) {
    int64_t p0 = ((int64_t)warp - off) % S;
    if (p0 < 0) p0 += S;
    for (int64_t p = p0 + (int64_t)lane * S; p < count; p += (int64_t)32 * S) {
      const unsigned char* rec = recs + p * rec_bytes;
      const int64_t idx = f64 ? reinterpret_cast<const int64_t*>(rec)[2] : (int64_t) reinterpret_cast<const int*>(rec)[4];
      const double m = reinterpret_cast<const double*>(rec)[1];
      if (REPRO) {
        const double hi = grid_round(m, obj[idx], gm);
        s += hi;
        s2 += grid_round(__fma_rn(m, obj[idx], -hi), 1.0, gm2);
      } else {
        s = fma(m, obj[idx], s);
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (REPRO)
    for (int o = 16; o > 0; o >>= 1) s2 += __shfl_down_sync(0xffffffffu, s2, o);
  if (lane == 0) out[warp] = s;
  if (REPRO && lane == 0) out2[warp] = s2;
}

int cell_objective(basq_ctx* ctx, const RecPool& pool, int64_t off_glob, int S, int S_eff, const double* obj,
                   double* out, double grid_m, double grid_m2, double* out2) {
  const int threads = 256;
  const int blocks = ceil_div((int64_t)S * 32, threads);
  if (grid_m != 0.0)
    cell_obj_kernel<true><<<blocks, threads, 0, ctx->stream>>>(pool.buf[pool.cur].as<unsigned char>(), pool.rec_bytes,
                                                               pool.dtype == BASQ_F64 ? 1 : 0, pool.count, off_glob, S,
                                                               S_eff, obj, out, grid_m, grid_m2, out2);
  else
    cell_obj_kernel<false><<<blocks, threads, 0, ctx->stream>>>(pool.buf[pool.cur].as<unsigned char>(), pool.rec_bytes,
                                                                pool.dtype == BASQ_F64 ? 1 : 0, pool.count, off_glob, S,
                                                                S_eff, obj, out, 0.0, 0.0, nullptr);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

// Maxima over the live records of |wf|, |mu| and |mu obj[idx]| (obj may be NULL: 0), the inputs of the grids of
// a reproducible pass.  out[3] must be zeroed; non-negative doubles order like their bit patterns.
__global__ void record_maxima_kernel(const unsigned char* __restrict__ recs, int rec_bytes, int f64, int64_t count,
                                     const double* __restrict__ obj, unsigned long long* __restrict__ out) {
  // NaN inputs: fmax would drop them, so !(x <= m) takes them over; a NaN bound makes session_set_grid fail
  auto take = [](double& m, double x) { if (!(x <= m)) m = x; };
  double m[3] = {0.0, 0.0, 0.0};
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < count; p += (int64_t)gridDim.x * blockDim.x) {
    const unsigned char* rec = recs + p * rec_bytes;
    const double* h = reinterpret_cast<const double*>(rec);
    if (m[0] == m[0]) take(m[0], fabs(h[0]));
    if (m[1] == m[1]) take(m[1], fabs(h[1]));
    if (obj && m[2] == m[2]) {
      const int64_t idx = f64 ? reinterpret_cast<const int64_t*>(rec)[2] : (int64_t) reinterpret_cast<const int*>(rec)[4];
      take(m[2], fabs(h[1] * obj[idx]));
    }
  }
  for (int i = 0; i < 3; ++i) {
    // a NaN becomes the canonical quiet NaN, whose bit pattern exceeds every non-negative double's
    double v = m[i] == m[i] ? m[i] : __longlong_as_double(0x7ff8000000000000ll);
    for (int o = 16; o > 0; o >>= 1) {
      const double u = __shfl_down_sync(0xffffffffu, v, o);
      if (__double_as_longlong(u) > __double_as_longlong(v)) v = u;
    }
    if ((threadIdx.x & 31) == 0) atomicMax(out + i, (unsigned long long)__double_as_longlong(v));
  }
}

int record_maxima(basq_ctx* ctx, const RecPool& pool, const double* obj, double* max_host) {
  DevBuf d;
  BASQ_TRY(d.alloc(ctx, 3 * sizeof(double)));
  BASQ_CUDA(cudaMemsetAsync(d.p, 0, 3 * sizeof(double), ctx->stream));
  if (pool.count > 0) {
    const int blocks = (int)std::min<int64_t>(ceil_div64(pool.count, 256), 4 * (int64_t)ctx->num_sms);
    record_maxima_kernel<<<blocks, 256, 0, ctx->stream>>>(pool.buf[pool.cur].as<unsigned char>(), pool.rec_bytes,
                                                          pool.dtype == BASQ_F64 ? 1 : 0, pool.count, obj,
                                                          d.as<unsigned long long>());
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
  }
  BASQ_CUDA(cudaMemcpyAsync(max_host, d.p, 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  BASQ_CUDA(cudaStreamSynchronize(ctx->stream));
  return BASQ_OK;
}

// ---------------------------------------------------------------------------------------------
// apply a round: mu *= omega[set] (and wf when it carries the measure), drop omega == 0, compact.
// Kept-point destination is analytic: D(g) = (g / S) * K + rank_excl[g % S]  (g = global position),
// so no scan is needed and the original order is preserved.
// One thread per 16-byte chunk of a record -> fully coalesced 16 B loads and stores.
// ---------------------------------------------------------------------------------------------
__global__ void apply_round_kernel(const unsigned char* __restrict__ src, unsigned char* __restrict__ dst,
                                   int chunks_per_rec, int64_t count, int64_t off, int S,
                                   const double* __restrict__ omega, const int* __restrict__ rank_excl, int K,
                                   int64_t dest_base, int scale_wf) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t p = t / chunks_per_rec;
  const int c = (int)(t - p * chunks_per_rec);
  if (p >= count) return;
  const int64_t g = off + p;
  const int j = (int)(g % S);
  const double om = omega[j];
  if (!(om > 0.0)) return;
  const int64_t dest = (g / S) * K + rank_excl[j] - dest_base;
  uint4 v = reinterpret_cast<const uint4*>(src)[p * chunks_per_rec + c];
  if (c == 0) {
    double wf = __hiloint2double((int)v.y, (int)v.x);
    double mu = __hiloint2double((int)v.w, (int)v.z);
    mu *= om;
    if (scale_wf) wf *= om;
    v.x = (unsigned)__double2loint(wf);
    v.y = (unsigned)__double2hiint(wf);
    v.z = (unsigned)__double2loint(mu);
    v.w = (unsigned)__double2hiint(mu);
  }
  reinterpret_cast<uint4*>(dst)[dest * chunks_per_rec + c] = v;
}

int apply_round(basq_ctx* ctx, RecPool* pool, int64_t off_glob, int S, const double* omega, const int* rank_excl,
                int K, bool scale_wf, int64_t dest_base, int64_t new_count) {
  BASQ_CHECK(new_count <= pool->capacity, BASQ_ERR_NUMERIC, "apply_round: %lld survivors exceed capacity %lld",
             (long long)new_count, (long long)pool->capacity);
  const int cpr = pool->rec_bytes / 16;
  const int64_t total = pool->count * cpr;
  if (total > 0) {
    const int threads = 256;
    const int64_t blocks = ceil_div64(total, threads);
    BASQ_CHECK(blocks < (1ll << 31), BASQ_ERR_UNSUPPORTED, "apply_round grid too large");
    apply_round_kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>(
        pool->buf[pool->cur].as<unsigned char>(), pool->buf[pool->cur ^ 1].as<unsigned char>(), cpr, pool->count,
        off_glob, S, omega, rank_excl, K, dest_base, scale_wf ? 1 : 0);
    ctx->launches++;
    BASQ_CUDA(cudaGetLastError());
  }
  pool->cur ^= 1;
  pool->count = new_count;
  return BASQ_OK;
}

// ---------------------------------------------------------------------------------------------
// result extraction
// ---------------------------------------------------------------------------------------------
__global__ void extract_kernel(const unsigned char* __restrict__ recs, int rec_bytes, int f64, int64_t count,
                               int64_t idx_base, int64_t* __restrict__ idx_out, double* __restrict__ w_out) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= count) return;
  const unsigned char* rec = recs + p * rec_bytes;
  w_out[p] = reinterpret_cast<const double*>(rec)[1];
  idx_out[p] = idx_base + (f64 ? reinterpret_cast<const int64_t*>(rec)[2] : (int64_t) reinterpret_cast<const int*>(rec)[4]);
}

int extract_result(basq_ctx* ctx, const RecPool& pool, int64_t idx_base, int64_t* idx_out, double* w_out) {
  if (pool.count == 0) return BASQ_OK;
  extract_kernel<<<ceil_div(pool.count, 256), 256, 0, ctx->stream>>>(pool.buf[pool.cur].as<unsigned char>(),
                                                                     pool.rec_bytes, pool.dtype == BASQ_F64 ? 1 : 0,
                                                                     pool.count, idx_base, idx_out, w_out);
  ctx->launches++;
  BASQ_CUDA(cudaGetLastError());
  return BASQ_OK;
}

}  // namespace basq
