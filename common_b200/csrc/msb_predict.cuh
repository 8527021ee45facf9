// msb_predict.cuh -- the posterior predictive of rows against the current suffstats (msb_state_predict): per row the log
// predictive density, the responsibilities and the MAP group, reduced from the score matrix the sweep's score kernels
// write (DESIGN.md section 4.9).  Every quantity is the sampler's own (util.hpp:125-136, DESIGN.md section 3):
//   m = max_c s_c,  p_c = msb_expf(s_c - m),  acc = sum_c p_c in fp64 in column order,
//   logp = m + log(acc) - log Z,  resp_c = RN(p_c / (float)acc),  MAP = the first column with s_c = m,
// where Z = sum_c pc_c (fp64) over the pseudocounts whose logs base_kernel adds to the columns.
#pragma once
#include "msb_score.cuh"

namespace msb {

// log Z: the pseudocounts of base_kernel (the group's count, or float(alpha / #empty) for an empty group) summed in fp64.
// One block.
__global__ void crp_logz_kernel(const double *__restrict__ counts, const int32_t *__restrict__ col2slot, int ncols,
                                float alpha, double *__restrict__ out) {
  __shared__ int s_empty;
  __shared__ double s_sum[32];
  if (threadIdx.x == 0) s_empty = 0;
  __syncthreads();
  int e = 0;
  for (int c = threadIdx.x; c < ncols; c += blockDim.x) e += counts[col2slot[c]] == 0.0;
  for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
  if ((threadIdx.x & 31) == 0 && e) atomicAdd(&s_empty, e);
  __syncthreads();
  const float per_empty = __fdiv_rn(alpha, (float)s_empty);
  double z = 0.0;
  for (int c = threadIdx.x; c < ncols; c += blockDim.x) {
    const double cnt = counts[col2slot[c]];
    z += (double)(cnt != 0.0 ? (float)cnt : per_empty);
  }
  for (int o = 16; o > 0; o >>= 1) z += __shfl_xor_sync(0xffffffffu, z, o);
  if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = z;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += s_sum[w];
    *out = log(t);
  }
}

// resp_c = RN(p / acc): Markstein's sequence where it equals the IEEE division (p = 0 or p >= 2^-100, acc in [1, 2^24];
// msb_kernels.cuh, dart_walk), __fdiv_rn elsewhere
__device__ __forceinline__ float resp_quotient(float p, float acc, float y) {
  return (acc >= 1.0f && acc <= 16777216.0f && (p == 0.f || p >= 0x1p-100f)) ? div_markstein(p, acc, y) : __fdiv_rn(p, acc);
}

__host__ __device__ inline size_t predict_tile_smem(int warps, int K, bool rowmajor) {
  return (size_t)warps * (sample_tile_bytes(K, rowmajor) + sizeof(uint64_t)) + 64;
}

// The 32-row tile form (K * 33 * 4 bytes fit, as for sample_tile_kernel): a warp stages the [K][32] tile of its 32 rows in
// shared memory -- one bulk copy of the blocked layout on an mbarrier, or transposing loads of a row-major one -- and then
//   pass 1  the row maximum, skipped where the score kernel's epilogue left it (rowmax);
//   pass 2  p = exp(s - m) a batch of eight groups at a time, chosen by a warp vote (dead: every x < -104 stores +0;
//           fast: every x in [-86, 0] runs msb_expf2_dense; else msb_expf), the in-order fp64 sum, and the first column
//           with x = s - m = 0 (the MAP: s - m rounds to 0 only for s = m);
//   pass 3  logp and the MAP column per lane; with resp, row by row, lanes over the groups: RN(p / acc) stored row-major,
//           coalesced, from a conflict-free transposed read of the tile.
// The blocked tile has pitch 32, so pass 2 stores p of (group k, row r) at k * 32 + (r ^ (k & 31)): the store (lanes over
// r) and pass 3's read (lanes over k) are both a permutation of the banks.  The row-major tile has pitch 33 and no swizzle.
template <int WARPS, bool ROWMAJOR>
__global__ void __launch_bounds__(WARPS * 32)
predict_tile_kernel(const float *__restrict__ scores, size_t ld, size_t skip, int K, size_t nrows, const int *__restrict__ rowmax,
                    const double *__restrict__ logz, double *__restrict__ logp, int32_t *__restrict__ map_col,
                    float *__restrict__ resp, size_t resp_ld) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int P = ROWMAJOR ? 33 : 32;
  const uint32_t tile_bytes = sample_tile_bytes(K, ROWMAJOR);
  const uint32_t copy_bytes = (uint32_t)K * 128u;
  float *tile = reinterpret_cast<float *>(smem_raw + (size_t)warp * tile_bytes);
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw + (size_t)WARPS * tile_bytes) + warp;
  auto pidx = [&](int k, int r) { return k * P + (ROWMAJOR ? r : (r ^ (k & 31))); };
  if (lane == 0) {
    mbar_init(smem_u32(bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  const double lz = *logz;
  const size_t blk_lo = skip / 32, blk_hi = (skip + nrows + 31) / 32;
  uint32_t parity = 0;
  for (size_t blk = blk_lo + (size_t)blockIdx.x * WARPS + warp; blk < blk_hi; blk += (size_t)gridDim.x * WARPS) {
    if constexpr (ROWMAJOR) {
      __syncwarp();
      for (int r = 0; r < 32; r++) {
        const long long ri = (long long)(blk * 32 + r) - (long long)skip;
        if (ri < 0 || (size_t)ri >= nrows) continue;
        const float *src = scores + (size_t)ri * ld;
        for (int kk = lane; kk < K; kk += 32) tile[kk * P + r] = src[kk];
      }
      __syncwarp();
    } else {
      if (lane == 0) {
        mbar_expect_tx(smem_u32(bar), copy_bytes);
        bulk_g2s(smem_u32(tile), scores + blk * ld * 32, copy_bytes, smem_u32(bar));
      }
      mbar_wait(smem_u32(bar), parity);
      parity ^= 1u;
    }
    const long long i = (long long)(blk * 32 + lane) - (long long)skip;
    const bool valid = i >= 0 && (size_t)i < nrows;
    const float *s = tile + lane;
    // pass 1
    float m = 0.f;
    bool scan = true;
    if (rowmax) {
      const int ord = rowmax[blk * 32 + lane];
      scan = ord == (int)0x80808080;
      m = ordered_float(ord);
    }
    if (__any_sync(0xffffffffu, scan)) {
      float m0 = s[0], m1 = m0, m2 = m0, m3 = m0;
      int k = 1;
      for (; k + 3 < K; k += 4) {
        m0 = fmaxf(m0, s[k * P]); m1 = fmaxf(m1, s[(k + 1) * P]);
        m2 = fmaxf(m2, s[(k + 2) * P]); m3 = fmaxf(m3, s[(k + 3) * P]);
      }
      for (; k < K; k++) m0 = fmaxf(m0, s[k * P]);
      if (scan) m = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
    }
    // pass 2
    double acc_d = 0.0;
    int map = -1;
    const float2 nm = make_float2(-m, -m);
    for (int k0 = 0; k0 < K; k0 += 8) {
      float x[8], p[8];
#pragma unroll
      for (int j = 0; j < 8; j += 2) {
        const float2 x2 = __fadd2_rn(make_float2(s[(k0 + j) * P], s[(k0 + j + 1) * P]), nm);
        x[j] = x2.x; x[j + 1] = x2.y;
      }
#pragma unroll
      for (int j = 0; j < 8; j++) {
        if (k0 + j >= K) x[j] = -CUDART_INF_F;
        if (map < 0 && x[j] == 0.f) map = k0 + j;
      }
      const float xhi = fmax8_nan(x);
      const bool dead = __all_sync(0xffffffffu, xhi < -104.0f);
      const float xlo = fmin8_nan(x);
      if (dead) {
#pragma unroll
        for (int j = 0; j < 8; j++) p[j] = 0.f;
      } else if (__all_sync(0xffffffffu, xlo >= -86.0f && xhi <= 0.0f)) {
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          const float2 p2 = msb_expf2_dense(make_float2(x[j], x[j + 1]));
          p[j] = p2.x; p[j + 1] = p2.y;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; j++) p[j] = msb_expf(x[j]);
      }
      if (!dead) {
#pragma unroll
        for (int j = 0; j < 8; j++) if (k0 + j < K) acc_d = __dadd_rn(acc_d, (double)p[j]);
      }
      if (resp) {
        if constexpr (!ROWMAJOR) __syncwarp();   // the swizzled stores overwrite scores of this batch that other lanes read
#pragma unroll
        for (int j = 0; j < 8; j++) tile[pidx(k0 + j, lane)] = p[j];
      }
    }
    // pass 3
    if (valid) {
      logp[i] = (double)m + log(acc_d) - lz;
      map_col[i] = map < 0 ? 0 : map;
    }
    if (resp) {
      const float acc = __double2float_rn(acc_d);
      __syncwarp();
      for (int r = 0; r < 32; r++) {
        const long long ri = (long long)(blk * 32 + r) - (long long)skip;
        const float a = __shfl_sync(0xffffffffu, acc, r);
        if (ri < 0 || (size_t)ri >= nrows) continue;
        const float y = __frcp_rn(a);
        float *dst = resp + (size_t)ri * resp_ld;
        for (int k = lane; k < K; k += 32) dst[k] = resp_quotient(tile[pidx(k, r)], a, y);
      }
    }
    if constexpr (!ROWMAJOR) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
  }
}

// The large-K form (the tile does not fit): one thread per row over the score matrix in global memory, as
// sample_blocked_kernel (blocked layout, rowmax from the epilogue) and sample_kernel (ROWMAJOR: the dm and CUDA-core NIW
// layouts) walk it.  Dead batches of eight groups (every x < -104 in every lane) are skipped in the sum; resp is staged
// through a 32 x 33 transpose per warp in shared memory so that its stores are coalesced.  Blocks of 128 threads.
template <bool ROWMAJOR>
__global__ void __launch_bounds__(128)
predict_rows_kernel(const float *__restrict__ scores, size_t ld, size_t skip, int K, size_t nrows, const int *__restrict__ rowmax,
                    const double *__restrict__ logz, double *__restrict__ logp, int32_t *__restrict__ map_col,
                    float *__restrict__ resp, size_t resp_ld) {
  __shared__ float tr[4][32][33];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < nrows;
  const size_t loc = (valid ? i : 0) + skip;
  const float *s = ROWMAJOR ? scores + (valid ? i : 0) * ld : scores + (loc / 32) * ld * 32 + (loc % 32);
  constexpr size_t STRIDE = ROWMAJOR ? 1 : 32;
  float m;
  const int ord = rowmax ? rowmax[loc] : (int)0x80808080;
  if (ord != (int)0x80808080) {
    m = ordered_float(ord);
  } else {
    float m0 = s[0], m1 = m0, m2 = m0, m3 = m0;
    int k = 1;
    for (; k + 3 < K; k += 4) {
      m0 = fmaxf(m0, s[k * STRIDE]); m1 = fmaxf(m1, s[(k + 1) * STRIDE]);
      m2 = fmaxf(m2, s[(k + 2) * STRIDE]); m3 = fmaxf(m3, s[(k + 3) * STRIDE]);
    }
    for (; k < K; k++) m0 = fmaxf(m0, s[k * STRIDE]);
    m = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
  }
  double acc_d = 0.0;
  int map = -1;
  for (int k0 = 0; k0 < K; k0 += 8) {
    float x[8];
    bool live = false;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      x[j] = k0 + j < K ? __fsub_rn(s[(size_t)(k0 + j) * STRIDE], m) : -CUDART_INF_F;
      live |= !exp_is_zero(x[j]);
    }
    if (!__any_sync(0xffffffffu, live)) continue;  // acc + 0 = acc, and no x = 0 in the batch
#pragma unroll
    for (int j = 0; j < 8; j++) {
      if (k0 + j >= K) continue;
      if (map < 0 && x[j] == 0.f) map = k0 + j;
      acc_d = __dadd_rn(acc_d, (double)msb_expf(x[j]));
    }
  }
  if (valid) {
    logp[i] = (double)m + log(acc_d) - *logz;
    map_col[i] = map < 0 ? 0 : map;
  }
  if (!resp) return;
  const float acc = __double2float_rn(acc_d);
  const float y = __frcp_rn(acc);
  const size_t row0 = (size_t)blockIdx.x * blockDim.x + warp * 32;
  for (int kc = 0; kc < K; kc += 32) {
#pragma unroll 4
    for (int j = 0; j < 32; j++) {
      const int k = kc + j;
      tr[warp][j][lane] = k < K ? resp_quotient(msb_expf(__fsub_rn(s[(size_t)k * STRIDE], m)), acc, y) : 0.f;
    }
    __syncwarp();
    for (int r = 0; r < 32; r++)
      if (row0 + r < nrows && kc + lane < K) resp[(row0 + r) * resp_ld + kc + lane] = tr[warp][lane][r];
    __syncwarp();
  }
}

}  // namespace msb
