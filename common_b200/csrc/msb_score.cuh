// msb_score.cuh -- the score kernel: N rows x K groups, summed over the scalar
// features (bb / dd / gp tables, nich closed form).
//
// Mapping (DESIGN.md "score kernel"):
//   * a block owns NW*RW rows and one k-tile of KT = 32*V groups;
//   * a warp owns RW rows; lane l owns V consecutive groups of the k-tile, so one
//     (row, feature) lookup is ONE conflict-free shared-memory wavefront per 32
//     groups and the row's value x is warp-uniform (shuffled from its owner lane);
//   * acc[RW][V] stays in registers across all features;
//   * the per-(feature, k-tile) parameter chunks are contiguous in global memory
//     in exactly the order the block consumes them, and are streamed through an
//     S-stage shared-memory ring with bulk async copies (cp.async.bulk, SASS
//     UBLKCP) completing on mbarriers -- no register staging, no __syncthreads
//     in the feature loop;
//   * the N x K result is written once with 128*V-byte coalesced stores.
#pragma once
#include <type_traits>

#include "msb_kernels.cuh"

namespace msb {

template <int V> struct VecF;
template <> struct VecF<1> { float v[1]; __device__ __forceinline__ void load(const float *p) { v[0] = *p; } };
template <> struct VecF<2> { float v[2]; __device__ __forceinline__ void load(const float *p) { const float2 t = *(const float2 *)p; v[0] = t.x; v[1] = t.y; } };
template <> struct VecF<4> { float v[4]; __device__ __forceinline__ void load(const float *p) { const float4 t = *(const float4 *)p; v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; } };

// the same loads from a 32-bit shared-memory address: the lookup address is then ONE integer multiply-add
// (per-lane chunk base + row index * row bytes) instead of the two the generic-pointer form compiles to
template <int V>
__device__ __forceinline__ void lds_vec(float *v, uint32_t addr) {
  if constexpr (V == 1) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v[0]) : "r"(addr));
  else if constexpr (V == 2) asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "r"(addr));
  else asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr));
}

template <int V>
__device__ __forceinline__ void store_vec(float *p, const float *a) {
  if constexpr (V == 1) *p = a[0];
  else if constexpr (V == 2) *(float2 *)p = make_float2(a[0], a[1]);
  else *(float4 *)p = make_float4(a[0], a[1], a[2], a[3]);
}

// compact per-feature record kept in shared memory by the score kernel
// which kernels keep thread 0 as the producer of the stage ring (see the end of the feature loop)
#ifndef MSB_FIXED_PRODUCER
#define MSB_FIXED_PRODUCER(tables_only) (tables_only)
#endif

struct FeatS {
  const uint32_t *scol;      // score column (u32 chunk-row index, or f32 value)
  const uint32_t *slowmask;  // per 32-row block bitmask of slow-path cells
  const void *col;           // value column (raw gp counts for the slow path)
  uint32_t rowoff;           // first chunk row inside the k-tile region
  uint32_t rows;             // chunk rows
  uint32_t ncat;
  uint16_t kind;
  uint16_t has_slow;
  uint32_t sx_off;           // score_bundle_kernel: offset of this feature's row values inside its stage
  uint32_t sc_off;           //                      offset of its parameter chunk
  uint32_t last;             //                      last feature of its bundle
  uint32_t fuse;             //                      first feature of a fused quad [bin, table, table, nich]
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// floats as integers that order the same way (an involution: applying it twice gives the float's bits back)
__device__ __forceinline__ int float_ordered(float f) {
  const int i = __float_as_int(f);
  return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float ordered_float(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// bounded wait: a protocol bug traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  // fast path: a phase that has already completed costs one try_wait, not a clock read as well
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  if (done) return;
  const long long t0 = clock64();
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}
// non-blocking: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
// global -> shared bulk copy (bytes % 16 == 0, both addresses 16-byte aligned), completes on bar
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// ---------------------------------------------------------------------------------------------------
// Sampler over the blocked score layout with the 32-row tile staged in shared memory: the tile
// ([K][32] floats, contiguous in global memory) is bulk-copied once and the three order-sensitive
// passes of util.hpp:125-156 (max / exp + double sum / dart scan) run from shared memory, lane = row,
// conflict-free.  exp(s - m) is computed once (pass 2 overwrites the tile with it).  HBM traffic: the
// score matrix is read exactly once.  Used when a tile fits (K * 128 bytes per warp).
// ---------------------------------------------------------------------------------------------------
// ROWMAJOR: the scores are row-major [row][ld] (the NIW kernels accumulate into that layout): the tile is filled
// by coalesced loads (lane = group) and stored transposed with pitch 33, conflict-free both ways.
// rowmax (may be null): the row maxima the score kernel's epilogue left (ordered integers, 0x80808080 where none was
// written); pass 1 then runs only for a warp with such a row.
//
// Shared memory per warp: the tile, K rounded up to 8 groups (pass 2 writes p = +0 into the padding, so the walk reads
// whole batches unconditionally), then one byte per (batch, lane): the biased exponent of the batch's largest p.
// Layout [WARPS tiles][WARPS mbarriers][WARPS exponent arrays]; sample_tile_smem() gives the size.
__host__ __device__ inline uint32_t sample_tile_bytes(int K, bool rowmajor) {
  return ((uint32_t)(K + 7) / 8u * 8u * (rowmajor ? 33u : 32u) * 4u + 127u) / 128u * 128u;
}
__host__ __device__ inline size_t sample_tile_smem(int warps, int K, bool rowmajor) {
  return (size_t)warps * (sample_tile_bytes(K, rowmajor) + sizeof(uint64_t) + (size_t)(K + 7) / 8 * 32) + 64;
}

// 3-input minimum / maximum (sm_100) that return NaN when an input is NaN
__device__ __forceinline__ float fmin3_nan(float a, float b, float c) {
  float d;
  asm("min.NaN.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ float fmax3_nan(float a, float b, float c) {
  float d;
  asm("max.NaN.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ float fmax8_nan(const float *v) {
  return fmax3_nan(fmax3_nan(v[0], v[1], v[2]), fmax3_nan(v[3], v[4], v[5]), fmax3_nan(v[6], v[7], v[7]));
}
__device__ __forceinline__ float fmin8_nan(const float *v) {
  return fmin3_nan(fmin3_nan(v[0], v[1], v[2]), fmin3_nan(v[3], v[4], v[5]), fmin3_nan(v[6], v[7], v[7]));
}

template <int WARPS, bool ROWMAJOR>
__global__ void __launch_bounds__(WARPS * 32)
sample_tile_kernel(const float *__restrict__ scores, size_t ld, size_t skip, int K, size_t nrows,
                   const float *__restrict__ uniforms, uint64_t seed, uint64_t sweep, uint64_t row_id0,
                   const int32_t *__restrict__ col2slot, int32_t *__restrict__ out_col, int32_t *__restrict__ out_slot,
                   const int *__restrict__ rowmax) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int P = ROWMAJOR ? 33 : 32;  // tile pitch in floats: element (group k, row r) at tile[k * P + r]
  const uint32_t tile_bytes = sample_tile_bytes(K, ROWMAJOR);
  const uint32_t copy_bytes = (uint32_t)K * 128u;   // the blocked layout's [K][32] tile
  const int nb = (K + 7) / 8;                        // batches of eight groups
  float *tile = reinterpret_cast<float *>(smem_raw + (size_t)warp * tile_bytes);
  uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw + (size_t)WARPS * tile_bytes) + warp;
  uint8_t *pexp = reinterpret_cast<uint8_t *>(smem_raw + (size_t)WARPS * (tile_bytes + sizeof(uint64_t))) +
                  (size_t)warp * nb * 32 + lane;
  if (lane == 0) {
    mbar_init(smem_u32(bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  const size_t blk_lo = skip / 32, blk_hi = (skip + nrows + 31) / 32;
  uint32_t parity = 0;
  for (size_t blk = blk_lo + (size_t)blockIdx.x * WARPS + warp; blk < blk_hi; blk += (size_t)gridDim.x * WARPS) {
    if constexpr (ROWMAJOR) {
      __syncwarp();
      for (int r = 0; r < 32; r++) {
        const long long ri = (long long)(blk * 32 + r) - (long long)skip;
        if (ri < 0 || (size_t)ri >= nrows) continue;
        const float *src = scores + (size_t)ri * ld;  // scores already points at the first valid row
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
    const long long i = (long long)(blk * 32 + lane) - (long long)skip;  // row of this lane, relative to the first valid row
    const bool valid = i >= 0 && (size_t)i < nrows;
    float *s = tile + lane;
    // pass 1: max (exact and order-independent: four partial maxima for instruction-level parallelism), unless the
    // score kernel left it: the same floats, the same maximum
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
    // pass 2: p = exp(s - m) (independent per k, kept in the tile) and the in-order double sum (the only chain),
    // a batch of eight groups at a time, chosen by a warp vote on its x = s - m:
    //   dead   every x < -104: every p is +0 (nothing to add to the sum, +0 stored)
    //   fast   every x in [-86, 0]: msb_expf2_dense, two groups per instruction (the same bits)
    //   else   msb_expf one group at a time (NaN, -inf, subnormal results)
    // and the biased exponent of the batch's largest p is recorded for the walk (NaN gives 255).
    double acc_d = 0.0;
    const float2 nm = make_float2(-m, -m);
    auto batch = [&](int k0, auto tail_tag) {
      constexpr bool TAIL = decltype(tail_tag)::value;
      float x[8], p[8];
#pragma unroll
      for (int j = 0; j < 8; j += 2) {  // s - m as s + (-m): the same rounding
        const float2 x2 = __fadd2_rn(make_float2(s[(k0 + j) * P], s[(k0 + j + 1) * P]), nm);
        x[j] = x2.x; x[j + 1] = x2.y;
      }
      if constexpr (TAIL) {
#pragma unroll
        for (int j = 0; j < 8; j++) if (k0 + j >= K) x[j] = -CUDART_INF_F;
      }
      const float xhi = fmax8_nan(x);
      if (__all_sync(0xffffffffu, xhi < -104.0f)) {
#pragma unroll
        for (int j = 0; j < 8; j++) s[(k0 + j) * P] = 0.f;
        pexp[(k0 >> 3) * 32] = 0;
        return;
      }
      const float xlo = fmin8_nan(x);
      if (__all_sync(0xffffffffu, xlo >= -86.0f && xhi <= 0.0f)) {
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          const float2 p2 = msb_expf2_dense(make_float2(x[j], x[j + 1]));
          p[j] = p2.x; p[j + 1] = p2.y;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; j++) p[j] = msb_expf(x[j]);
      }
#pragma unroll
      for (int j = 0; j < 8; j++) {
        s[(k0 + j) * P] = p[j];
        if (!TAIL || k0 + j < K) acc_d = __dadd_rn(acc_d, (double)p[j]);
      }
      pexp[(k0 >> 3) * 32] = (uint8_t)(__float_as_uint(fmax8_nan(p)) >> 23);
    };
    const int kfull = K & ~7;
    for (int k0 = 0; k0 < kfull; k0 += 8) batch(k0, std::false_type{});
    if (kfull < K) batch(kfull, std::true_type{});
    const float acc = __double2float_rn(acc_d);
    float dart = 0.f;
    if (valid) dart = uniforms ? uniforms[i] : philox_u01(seed, row_id0 + (uint64_t)i, sweep);
    // pass 3: the dart walk (msb_kernels.cuh), quotients from the tile.  A lane whose dart d >= 2^-60 is normal keeps
    // d bit for bit over a batch whose every q = RN(p / acc) is below h = 2^(floor(log2 d) - 25) -- at most half the
    // spacing of the floats just below d, so RN(d - q) = d -- and then makes no pick either (d stays > 0).  With
    // E the batch's recorded exponent (every p < 2^(E - 126)) and acc in [1, 2^24] (acc >= 2^(Ea - 127)),
    //   E <= Ea + Ed - 154  gives  p / acc < 2^(Ed - 153) = h / 2,  so  RN(p / acc) <= pred(h) < h
    // (Ea, Ed: biased exponents of acc and d; E = 255 for a NaN p never passes).  Such a batch is skipped when every
    // lane still walking passes; the exact conditions are in DESIGN.md section 4.3.
    int pick;
    dart_walk<true>(K, acc, dart, !valid, pick, [&](int kk) { return s[kk * P]; },
                    [&](int k0, bool f, float d) { return f || dart_keeps(pexp[(k0 >> 3) * 32], acc, d); });
    if (valid) {
      if (out_col) out_col[i] = pick;
      if (out_slot) out_slot[i] = col2slot ? col2slot[pick] : pick;
    }
    // the next bulk copy (async proxy) overwrites the tile this warp has just read and written (generic proxy)
    if constexpr (!ROWMAJOR) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
  }
}

// gp count beyond the lookup table: fp64 closed form straight from the suffstats.  Kept out of line so
// that its fp64 register pressure stays off the hot loop.
__device__ __noinline__ float gp_overflow_score(const FeatDev *f, const double *hp, const double *ss, int slot, double xv) {
  const double *h = hp + f->hp_off, *g = ss + f->ss_off + (size_t)slot * f->ss_w;
  return f->family == FAM_BNB ? (float)bnb_score(bnb_post(h, g), xv) : (float)gp_score(gp_post(h, g), xv);
}

// Output layouts of the N x K score matrix:
//   row-major   scores[(row - row_org) * ld + col]                     (the API's observable output)
//   blocked     scores[((row - row_org) / 32 * ld + col) * 32 + (row - row_org) % 32]
//               32-row blocks, group-major inside a block: the sampler walks one row per thread and
//               reads it fully coalesced.  Internal to the sweep.
// row_org (a multiple of 128, <= row_lo) is the first row the grid covers; rows < row_lo are not written.
// TABLES_ONLY: every feature is a lookup table without slow-path cells: no kind dispatch at all.
//
// Stage layout (one per feature in flight): [row values: NW*RW u32][slow masks: NW*RW/32 u32][pad to 128][chunk]
template <int V, int RW, int NW, bool BLOCKED, bool TABLES_ONLY>
__global__ void __launch_bounds__(NW * 32, 1)
score_kernel(const FeatDev *__restrict__ feats, int nfeat, const float *__restrict__ params, size_t region_rows,
             uint32_t stage_bytes, int S, const float *__restrict__ base, float *__restrict__ scores, size_t ld,
             size_t row_org, size_t row_lo, size_t row_hi, const double *__restrict__ hp,
             const double *__restrict__ ss, const int32_t *__restrict__ col2slot, int ncols, int ktiles, int tail_g,
             int *__restrict__ rowmax) {
  constexpr int KT = 32 * V;
  constexpr int RL = RW / 32;
  constexpr int RB = NW * RW;                                   // rows per block
  constexpr uint32_t X_BYTES = RB * 4, M_BYTES = RB / 8;        // row values, slow masks
  constexpr uint32_t CHUNK_OFF = (X_BYTES + M_BYTES + 127) / 128 * 128;
  static_assert(RW % 32 == 0 && M_BYTES % 16 == 0, "tile sizes must keep the bulk copies 16-byte granular");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // layout: [S stages | mbarriers full[S], empty[S] | feature table]
  unsigned char *stages = smem_raw;
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)S * stage_bytes);
  FeatS *ftab = reinterpret_cast<FeatS *>(bars + 2 * S);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // 1-D grid, k-tile fastest: the blocks that share a row tile run together, so its row values come
  // from DRAM once and from L2 for the other k-tiles
  const int kt = (int)(blockIdx.x % (unsigned)ktiles);
  const float *region = params + (size_t)kt * region_rows * KT;
  const size_t blk_row0 = row_org + (size_t)(blockIdx.x / (unsigned)ktiles) * RB;   // multiple of 128
  const size_t row0 = blk_row0 + (size_t)warp * RW;

  for (int i = tid; i < nfeat; i += NW * 32) {
    const FeatDev f = feats[i];
    FeatS t;
    t.scol = f.scol; t.slowmask = f.slowmask; t.col = f.col;
    t.rowoff = f.rowoff; t.rows = f.rows; t.ncat = f.ncat;
    t.kind = (uint16_t)((f.kind == KIND_TABLE && f.binform) ? KIND_BIN : f.kind); t.has_slow = (uint16_t)(f.has_slow != 0);
    t.sx_off = t.sc_off = 0; t.last = 1; t.fuse = 0;
    ftab[i] = t;
  }
  if (tid == 0) {
    for (int s = 0; s < S; s++) {
      mbar_init(smem_u32(&bars[s]), 1);
      if constexpr (MSB_FIXED_PRODUCER(TABLES_ONLY)) mbar_init(smem_u32(&bars[S + s]), NW);
      else bars[S + s] = 0;  // release counter of the stage (see the end of the feature loop)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // one thread: everything feature d needs -> stage s (row values, slow masks, parameter chunk)
  auto issue = [&](int d, int s) {
    const FeatS t = ftab[d];
    const uint32_t cbytes = t.rows * (uint32_t)(KT * sizeof(float));
    const uint32_t bar = smem_u32(&bars[s]);
    const uint32_t dst = smem_u32(stages + (size_t)s * stage_bytes);
    const bool slow = !TABLES_ONLY && t.has_slow;
    mbar_expect_tx(bar, cbytes + X_BYTES + (slow ? M_BYTES : 0u));
    bulk_g2s(dst, t.scol + blk_row0, X_BYTES, bar);
    if (slow) bulk_g2s(dst + X_BYTES, t.slowmask + (blk_row0 >> 5), M_BYTES, bar);
    bulk_g2s(dst + CHUNK_OFF, region + (size_t)t.rowoff * KT, cbytes, bar);
  };
  if (tid == 0)
    for (int d = 0; d < S && d < nfeat; d++) issue(d, d);

  // Ragged last k-tile (V = 1, tables only): when it holds tail_g <= 16 groups, build_params_kernel replicates its
  // table columns 32 / tail_g times across the 32-float chunk row, and lane l owns group l % tail_g of the rows
  // r = l / tail_g (mod 32 / tail_g): one conflict-free wavefront then serves 32 / tail_g rows instead of one
  // (C2: K = 200 = 6 x 32 + 8, the 7th tile costs ~45 % of a full one).  acc[s][0] holds row (32 / tail_g) s + l / tail_g.
  const bool tail = V == 1 && TABLES_ONLY && tail_g > 0 && kt == ktiles - 1;

  float acc[RW][V];
#pragma unroll
  for (int r = 0; r < RW; r++)
#pragma unroll
    for (int v = 0; v < V; v++) acc[r][v] = 0.f;

  int s = 0;
  uint32_t parity = 0;
  for (int d = 0; d < nfeat; d++) {
    const FeatS t = ftab[d];
    mbar_wait(smem_u32(&bars[s]), parity);
    const unsigned char *st = stages + (size_t)s * stage_bytes;
    // this warp's RW row values, read as broadcast 128-bit loads (4 rows per shared-memory wavefront)
    const uint4 *xq = reinterpret_cast<const uint4 *>(st) + warp * (RW / 4);
    const float *chunk = reinterpret_cast<const float *>(st + CHUNK_OFF) + lane * V;
    uint32_t slow[RL];
#pragma unroll
    for (int j = 0; j < RL; j++)
      slow[j] = (!TABLES_ONLY && t.has_slow) ? reinterpret_cast<const uint32_t *>(st + X_BYTES)[warp * RL + j] : 0u;

    if (V == 1 && TABLES_ONLY && tail) {
      const uint32_t chunk_s = smem_u32(chunk);
      auto tail_lookup = [&](auto rtag) {
        constexpr int R = decltype(rtag)::value;  // rows per wavefront
        const uint32_t *xw = reinterpret_cast<const uint32_t *>(st) + warp * RW + lane / (32 / R);
#pragma unroll
        for (int q = 0; q < RW / R; q++) {
          float tv[1];
          lds_vec<1>(tv, chunk_s + xw[q * R] * (uint32_t)(KT * sizeof(float)));
          acc[q][0] += tv[0];
        }
      };
      if (tail_g == 8) tail_lookup(std::integral_constant<int, 4>{});
      else tail_lookup(std::integral_constant<int, 2>{});
    } else if (!TABLES_ONLY && t.kind == KIND_BIN) {  // bb in binary form: acc += x (t1 - t0), sum_d t0 is already in base[]
      VecF<V> df;
      df.load(chunk + 0 * KT);
#pragma unroll
      for (int r4 = 0; r4 < RW / 4; r4++) {
        const uint4 q = xq[r4];
        const float xs[4] = {__uint_as_float(q.x), __uint_as_float(q.y), __uint_as_float(q.z), __uint_as_float(q.w)};
#pragma unroll
        for (int e = 0; e < 4; e++) {
          if constexpr (V % 2 == 0) {
#pragma unroll
            for (int h = 0; h < V / 2; h++) {
              const float2 a = __ffma2_rn(make_float2(xs[e], xs[e]), make_float2(df.v[2 * h], df.v[2 * h + 1]),
                                          make_float2(acc[r4 * 4 + e][2 * h], acc[r4 * 4 + e][2 * h + 1]));
              acc[r4 * 4 + e][2 * h] = a.x;
              acc[r4 * 4 + e][2 * h + 1] = a.y;
            }
          } else {
#pragma unroll
            for (int v = 0; v < V; v++) acc[r4 * 4 + e][v] = fmaf(xs[e], df.v[v], acc[r4 * 4 + e][v]);
          }
        }
      }
      // masked cells were scored as x = 0: take back the t0 that base[] carries for this feature (rare)
#pragma unroll
      for (int j = 0; j < RL; j++) {
        uint32_t m = slow[j];
        if (m) {
          VecF<V> t0;
          t0.load(chunk + 1 * KT);
          while (m) {
            const int rr = j * 32 + __ffs(m) - 1;
            m &= m - 1;
#pragma unroll
            for (int r = 0; r < RW; r++)
              if (r == rr)
#pragma unroll
                for (int v = 0; v < V; v++) acc[r][v] -= t0.v[v];
          }
        }
      }
    } else if (TABLES_ONLY || t.kind != KIND_NICH) {
      const uint32_t chunk_s = smem_u32(chunk);
#pragma unroll
      for (int r4 = 0; r4 < RW / 4; r4++) {
        const uint4 q = xq[r4];
        const uint32_t idx[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < 4; e++) {
          VecF<V> tv;
          lds_vec<V>(tv.v, chunk_s + idx[e] * (uint32_t)(KT * sizeof(float)));
          if constexpr (V % 2 == 0) {
#pragma unroll
            for (int h = 0; h < V / 2; h++) {
              const float2 a = __fadd2_rn(make_float2(acc[r4 * 4 + e][2 * h], acc[r4 * 4 + e][2 * h + 1]),
                                          make_float2(tv.v[2 * h], tv.v[2 * h + 1]));
              acc[r4 * 4 + e][2 * h] = a.x;
              acc[r4 * 4 + e][2 * h + 1] = a.y;
            }
          } else {
#pragma unroll
            for (int v = 0; v < V; v++) acc[r4 * 4 + e][v] += tv.v[v];
          }
        }
      }
      if (!TABLES_ONLY && t.kind == KIND_GP) {  // counts beyond the table: the fp64 closed form from the suffstats (rare)
        const uint32_t *raw = reinterpret_cast<const uint32_t *>(t.col);
#pragma unroll
        for (int j = 0; j < RL; j++) {
          uint32_t m = slow[j];
          while (m) {
            const int rr = j * 32 + __ffs(m) - 1;
            m &= m - 1;
            const double xv = (double)raw[row0 + rr];
            float add[V];
#pragma unroll
            for (int v = 0; v < V; v++) {
              const int col = kt * KT + lane * V + v;
              add[v] = 0.f;
              if (col < ncols) add[v] = gp_overflow_score(feats + d, hp, ss, col2slot[col], xv);
            }
#pragma unroll
            for (int r = 0; r < RW; r++)  // static register indexing: acc must not spill to local memory
              if (r == rr)
#pragma unroll
                for (int v = 0; v < V; v++) acc[r][v] += add[v];
          }
        }
      }
    } else {  // KIND_NICH: c1' log2(1 + ((x - mu) s)^2); sum_d c0 is already in base[]
      VecF<V> mu, sc, c1;
      mu.load(chunk + 0 * KT);
      sc.load(chunk + 1 * KT);
      c1.load(chunk + 2 * KT);
      if constexpr (V % 2 == 0) {  // two groups per instruction (FADD2 / FMUL2 / FFMA2)
        float2 nmu2[V / 2], sc2[V / 2], c12[V / 2];
#pragma unroll
        for (int h = 0; h < V / 2; h++) {
          nmu2[h] = make_float2(-mu.v[2 * h], -mu.v[2 * h + 1]);
          sc2[h] = make_float2(sc.v[2 * h], sc.v[2 * h + 1]);
          c12[h] = make_float2(c1.v[2 * h], c1.v[2 * h + 1]);
        }
#pragma unroll
        for (int r4 = 0; r4 < RW / 4; r4++) {
          const uint4 q = xq[r4];
          const float xs[4] = {__uint_as_float(q.x), __uint_as_float(q.y), __uint_as_float(q.z), __uint_as_float(q.w)};
#pragma unroll
          for (int e = 0; e < 4; e++) {
            const float2 x2 = make_float2(xs[e], xs[e]);
#pragma unroll
            for (int h = 0; h < V / 2; h++) {
              const float2 tt = __fmul2_rn(__fadd2_rn(x2, nmu2[h]), sc2[h]);
              const float2 a = __ffma2_rn(c12[h], log2_1p_pos2(__fmul2_rn(tt, tt)),
                                          make_float2(acc[r4 * 4 + e][2 * h], acc[r4 * 4 + e][2 * h + 1]));
              acc[r4 * 4 + e][2 * h] = a.x;
              acc[r4 * 4 + e][2 * h + 1] = a.y;
            }
          }
        }
      } else {
#pragma unroll
        for (int r4 = 0; r4 < RW / 4; r4++) {
          const uint4 q = xq[r4];
          const float xs[4] = {__uint_as_float(q.x), __uint_as_float(q.y), __uint_as_float(q.z), __uint_as_float(q.w)};
#pragma unroll
          for (int e = 0; e < 4; e++)
#pragma unroll
            for (int v = 0; v < V; v++) {
              const float tt = (xs[e] - mu.v[v]) * sc.v[v];
              acc[r4 * 4 + e][v] = fmaf(c1.v[v], log2_1p_pos(tt * tt), acc[r4 * 4 + e][v]);
            }
        }
      }
      // masked cells were scored as x = 0: undo that term and the c0 that base[] carries for this feature (rare)
#pragma unroll
      for (int j = 0; j < RL; j++) {
        uint32_t m = slow[j];
        if (m) {
          VecF<V> c0;
          c0.load(chunk + 3 * KT);
          float undo[V];
#pragma unroll
          for (int v = 0; v < V; v++) {
            const float tt = (0.f - mu.v[v]) * sc.v[v];
            undo[v] = -fmaf(c1.v[v], log2_1p_pos(tt * tt), c0.v[v]);
          }
          while (m) {
            const int rr = j * 32 + __ffs(m) - 1;
            m &= m - 1;
#pragma unroll
            for (int r = 0; r < RW; r++)
              if (r == rr)
#pragma unroll
                for (int v = 0; v < V; v++) acc[r][v] += undo[v];
          }
        }
      }
    }
    // Release the stage; the refill with feature d + S is issued once every warp has released it.
    __syncwarp();
    if constexpr (MSB_FIXED_PRODUCER(TABLES_ONLY)) {
      // thread 0 is the producer: it waits for the other warps' releases, then issues the copies
      if (lane == 0) mbar_arrive(smem_u32(&bars[S + s]));
      if (tid == 0 && d + S < nfeat) {
        mbar_wait(smem_u32(&bars[S + s]), parity);
        issue(d + S, s);
      }
    } else {
      // A release counter per stage, and the warp that arrives LAST issues the refill: nobody waits here.  With thread 0
      // as the fixed producer, warp 0 -- which cannot go on before the slowest warp has finished the feature -- falls
      // behind by construction; with 8 warps of long arithmetic chains the others then run S features ahead into a
      // stage that is only just being requested (ncu: 9 % of the samples on the full-barrier spin).  C3 93.7 -> 87.4 ms,
      // C5 47.5 -> 44.0 ms.  The tables-only kernel keeps the fixed producer: measured, it is the faster of the two there
      // (C2 1.40 against 1.46 ms).  Also measured and not kept: looking at the counter's return value one feature
      // later, so that no warp waits for the atomic (C2 1.48, C3 87.3, C5 46.2 ms), and a producer role that rotates
      // over the warps (C2 1.44, C3 97.1, C5 50.8 ms).
      if (lane == 0) {
        // acq_rel: this warp's reads of the stage (ordered before lane 0 by the __syncwarp above) happen before the
        // increment, and the last arriver's refill happens after every other warp's increment
        const uint32_t rel = smem_u32(&bars[S + s]);
        unsigned int old;
        asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(rel) : "memory");
        if (old == (unsigned)(NW - 1)) {
          // nobody touches the counter again before the refill below has landed and been consumed
          asm volatile("st.relaxed.cta.shared::cta.u32 [%0], %1;" ::"r"(rel), "r"(0u) : "memory");
          if (d + S < nfeat) issue(d + S, s);
        }
      }
    }
    if (++s == S) { s = 0; parity ^= 1u; }
  }

  // epilogue: + log(pseudocount) (group_manager.hpp:274-283)
  if (V == 1 && TABLES_ONLY && tail) {
    auto tail_epilogue = [&](auto rtag) {
      constexpr int R = decltype(rtag)::value;  // rows per wavefront; this lane: rows R q + sub, group g
      constexpr int G = 32 / R;
      const int sub = lane / G, g = lane % G;
      const float bg = base[(size_t)kt * KT + g];
      if constexpr (!BLOCKED) {
#pragma unroll
        for (int q = 0; q < RW / R; q++) {
          const size_t row = row0 + (size_t)q * R + sub;
          if (row >= row_lo && row < row_hi) scores[(row - row_org) * ld + (size_t)kt * KT + g] = acc[q][0] + bg;
        }
      } else {
        __syncthreads();  // every warp has finished reading the stages
        float *tile = reinterpret_cast<float *>(stages) + (size_t)warp * 32 * (KT + 1);
#pragma unroll
        for (int j = 0; j < RL; j++) {
          __syncwarp();
#pragma unroll
          for (int q = 0; q < G; q++) tile[(q * R + sub) * (KT + 1) + g] = acc[j * G + q][0] + bg;
          __syncwarp();
          const size_t rb = (row0 - row_org) / 32 + j;
          if (row0 + (size_t)j * 32 < row_hi) {
            float *dst = scores + (rb * ld + (size_t)kt * KT) * 32 + lane;
            float mx = -CUDART_INF_F;
#pragma unroll
            for (int c = 0; c < G; c++) {
              const float v = tile[lane * (KT + 1) + c];
              dst[(size_t)c * 32] = v;
              if (kt * KT + c < ncols) mx = fmaxf(mx, v);
            }
            if (rowmax) atomicMax(rowmax + rb * 32 + lane, float_ordered(mx));
          }
        }
      }
    };
    if (tail_g == 8) tail_epilogue(std::integral_constant<int, 4>{});
    else tail_epilogue(std::integral_constant<int, 2>{});
    return;
  }
  VecF<V> b;
  b.load(base + (size_t)kt * KT + lane * V);
  if constexpr (!BLOCKED) {  // 128 V-byte coalesced row-major stores
#pragma unroll
    for (int r = 0; r < RW; r++) {
      const size_t row = row0 + r;
      if (row >= row_lo && row < row_hi) {
        float o[V];
#pragma unroll
        for (int v = 0; v < V; v++) o[v] = acc[r][v] + b.v[v];
        store_vec<V>(scores + (row - row_org) * ld + (size_t)kt * KT + lane * V, o);
      }
    }
  } else {
    // transpose each 32-row x KT-group tile through shared memory (the drained stage ring) so that
    // lane = row and every store instruction writes 32 consecutive floats of one group
    __syncthreads();  // every warp has finished reading the stages
    float *tile = reinterpret_cast<float *>(stages) + (size_t)warp * 32 * (KT + 1);
#pragma unroll
    for (int j = 0; j < RL; j++) {
      __syncwarp();
#pragma unroll
      for (int r = 0; r < 32; r++)
#pragma unroll
        for (int v = 0; v < V; v++) tile[r * (KT + 1) + lane * V + v] = acc[j * 32 + r][v] + b.v[v];
      __syncwarp();
      const size_t rb = (row0 - row_org) / 32 + j;
      if (row0 + (size_t)j * 32 < row_hi) {
        float *dst = scores + (rb * ld + (size_t)kt * KT) * 32 + lane;
        // the row's largest score over this k-tile's real groups goes to the sampler, as in score_bundle_kernel
        float mx = -CUDART_INF_F;
#pragma unroll 8
        for (int c = 0; c < KT; c++) {
          const float v = tile[lane * (KT + 1) + c];
          dst[(size_t)c * 32] = v;
          if (kt * KT + c < ncols) mx = fmaxf(mx, v);
        }
        if (rowmax) atomicMax(rowmax + rb * 32 + lane, float_ordered(mx));
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// score_tables_persistent_kernel -- the sweep's tables-only score kernel (every feature a lookup table, no slow-path
// cells, blocked output), one CTA per SM for the whole launch.
//
// Same mapping as score_kernel<V, RW, NW, true, true> (a warp owns RW rows, lane l owns V groups of the k-tile, one
// conflict-free wavefront per lookup), but the CTA walks work items (row tile, k-tile) -- item = blockIdx.x + j gridDim.x,
// k-tile fastest, so the CTAs running together share row tiles through L2 exactly as the one-item-per-block grid did --
// and the stage ring runs THROUGH the item boundaries: while the warps of an item add the log-prior and store, the
// copies of the next item's first S features are already in flight.  The epilogue stores straight from registers (see
// there), so it needs no block-wide barrier, no drained ring and no transposition buffer.  ncu on the
// one-item-per-block kernel (C2, profiles/r01_prof_score_r1j_C2.txt) put ~13 % of the warp samples on block
// boundaries: the launch of 6839 blocks of 512 threads, the feature-table build, the first stage's latency, the
// __syncthreads before the transposition, the ring idle during the stores.
// ---------------------------------------------------------------------------------------------------
template <int V, int RW, int NW>
__global__ void __launch_bounds__((NW + 1) * 32, 1)
score_tables_persistent_kernel(const FeatDev *__restrict__ feats, int nfeat, const float *__restrict__ params, size_t region_rows,
                               uint32_t stage_bytes, int S, const float *__restrict__ base, float *__restrict__ scores, size_t ld,
                               size_t row_org, size_t row_lo, size_t row_hi, int ktiles, int tail_g, long long n_items) {
  constexpr int KT = 32 * V;
  constexpr int RL = RW / 32;
  constexpr int RB = NW * RW;                                   // rows per item
  constexpr uint32_t X_BYTES = RB * 4;                          // row values
  constexpr uint32_t CHUNK_OFF = (X_BYTES + RB / 8 + 127) / 128 * 128;   // the stage layout of score_kernel (no slow masks here)
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // layout: [S stages | mbarriers full[S], empty[S] | feature table]
  unsigned char *stages = smem_raw;
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)S * stage_bytes);
  FeatS *ftab = reinterpret_cast<FeatS *>(bars + 2 * S);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  for (int i = tid; i < nfeat; i += (NW + 1) * 32) {
    const FeatDev f = feats[i];
    FeatS t;
    t.scol = f.scol; t.slowmask = f.slowmask; t.col = f.col;
    t.rowoff = f.rowoff; t.rows = f.rows; t.ncat = f.ncat;
    t.kind = (uint16_t)f.kind; t.has_slow = 0;
    t.sx_off = t.sc_off = 0; t.last = 1; t.fuse = 0;
    ftab[i] = t;
  }
  if (tid == 0) {
    for (int s = 0; s < S; s++) {
      mbar_init(smem_u32(&bars[s]), 1);
      mbar_init(smem_u32(&bars[S + s]), NW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  const long long my_items = n_items > (long long)blockIdx.x ? (n_items - 1 - (long long)blockIdx.x) / (long long)gridDim.x + 1 : 0;
  const long long nq = my_items * nfeat;   // (item, feature) pairs this CTA walks, in order

  // item -> (row tile, k-tile) without a division per step: the CTA's items advance by gridDim.x
  const int dk = (int)(gridDim.x % (unsigned)ktiles);
  const size_t dr = gridDim.x / (unsigned)ktiles;
  // thread 0: everything the next (item, feature) pair needs -> stage s (row values, parameter chunk)
  int iss_d = 0, iss_kt = (int)(blockIdx.x % (unsigned)ktiles);
  size_t iss_rt = blockIdx.x / (unsigned)ktiles;
  auto issue_next = [&](int s) {
    const FeatS t = ftab[iss_d];
    const uint32_t cbytes = t.rows * (uint32_t)(KT * sizeof(float));
    const uint32_t bar = smem_u32(&bars[s]);
    const uint32_t dst = smem_u32(stages + (size_t)s * stage_bytes);
    mbar_expect_tx(bar, cbytes + X_BYTES);
    bulk_g2s(dst, t.scol + (row_org + iss_rt * RB), X_BYTES, bar);
    bulk_g2s(dst + CHUNK_OFF, params + ((size_t)iss_kt * region_rows + t.rowoff) * KT, cbytes, bar);
    if (++iss_d == nfeat) {
      iss_d = 0;
      iss_kt += dk; iss_rt += dr;
      if (iss_kt >= ktiles) { iss_kt -= ktiles; iss_rt++; }
    }
  };
  if (warp == NW) {
    // ===== producer warp: one lane keeps the ring full -- the first S pairs at once, then pair q into its stage as soon
    // as every consumer warp has released pair q - S.  A consumer thread doing this on the side (thread 0 of the
    // one-item-per-block kernel) has to wait for the slowest warp of every feature before it goes on with its own
    // lookups: warp 0 becomes the laggard of the block and the others run S features ahead, then wait for it.
    if (lane == 0) {
      int rs = 0;
      uint32_t rpar = 1;   // parity of the release awaited: 0 during the ring's second round, then alternating
      for (long long q = 0; q < nq; q++) {
        if (q >= S) mbar_wait(smem_u32(&bars[S + rs]), rpar);
        issue_next(rs);
        if (++rs == S) { rs = 0; rpar ^= 1u; }
      }
    }
    return;
  }

  int s = 0;
  uint32_t parity = 0;
  int kt = (int)(blockIdx.x % (unsigned)ktiles);
  size_t rt = blockIdx.x / (unsigned)ktiles;
  for (long long it = 0; it < my_items; it++) {
    if (it) {
      kt += dk; rt += dr;
      if (kt >= ktiles) { kt -= ktiles; rt++; }
    }
    const size_t row0 = row_org + rt * RB + (size_t)warp * RW;
    // Ragged last k-tile (V = 1): when it holds tail_g <= 16 groups, build_params_kernel replicates its table columns
    // 32 / tail_g times across the chunk row, and lane l owns group l % tail_g of the rows r = l / tail_g (mod 32 / tail_g):
    // one wavefront then serves 32 / tail_g rows (see score_kernel)
    const bool tail = V == 1 && tail_g > 0 && kt == ktiles - 1;

    float acc[RW][V];
#pragma unroll
    for (int r = 0; r < RW; r++)
#pragma unroll
      for (int v = 0; v < V; v++) acc[r][v] = 0.f;

    for (int d = 0; d < nfeat; d++) {
      mbar_wait(smem_u32(&bars[s]), parity);
      const unsigned char *st = stages + (size_t)s * stage_bytes;
      const uint4 *xq = reinterpret_cast<const uint4 *>(st) + warp * (RW / 4);
      const uint32_t chunk_s = smem_u32(reinterpret_cast<const float *>(st + CHUNK_OFF) + lane * V);
      if (V == 1 && tail) {
        auto tail_lookup = [&](auto rtag) {
          constexpr int R = decltype(rtag)::value;  // rows per wavefront
          const uint32_t *xw = reinterpret_cast<const uint32_t *>(st) + warp * RW + lane / (32 / R);
#pragma unroll
          for (int q = 0; q < RW / R; q++) {
            float tv[1];
            lds_vec<1>(tv, chunk_s + xw[q * R] * (uint32_t)(KT * sizeof(float)));
            acc[q][0] += tv[0];
          }
        };
        if (tail_g == 8) tail_lookup(std::integral_constant<int, 4>{});
        else tail_lookup(std::integral_constant<int, 2>{});
      } else {
#pragma unroll
        for (int r4 = 0; r4 < RW / 4; r4++) {
          const uint4 q = xq[r4];
          const uint32_t idx[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
          for (int e = 0; e < 4; e++) {
            VecF<V> tv;
            lds_vec<V>(tv.v, chunk_s + idx[e] * (uint32_t)(KT * sizeof(float)));
            if constexpr (V % 2 == 0) {
#pragma unroll
              for (int h = 0; h < V / 2; h++) {
                const float2 a = __fadd2_rn(make_float2(acc[r4 * 4 + e][2 * h], acc[r4 * 4 + e][2 * h + 1]),
                                            make_float2(tv.v[2 * h], tv.v[2 * h + 1]));
                acc[r4 * 4 + e][2 * h] = a.x;
                acc[r4 * 4 + e][2 * h + 1] = a.y;
              }
            } else {
#pragma unroll
              for (int v = 0; v < V; v++) acc[r4 * 4 + e][v] += tv.v[v];
            }
          }
        }
      }
      // release the stage: the producer warp refills it once every consumer warp has released it
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bars[S + s]));
      if (++s == S) { s = 0; parity ^= 1u; }
    }

    // epilogue: + log(pseudocount) (group_manager.hpp:274-283).  No transposition: in the blocked layout the 32 rows of
    // one (row block, group) are 128 contiguous bytes, and a lane already holds all the rows of its V groups -- it
    // writes them itself, eight 16-byte stores per (row block, group).  A warp's store instruction then touches 32 lines
    // (16 bytes each; the next instruction completes the sectors, L2 merges them), twice the write requests of the
    // transposed form, but no shared-memory round trip (2 x 128 KB of wavefronts per item) and no tile buffers: the
    // ring keeps all of shared memory.
    if (V == 1 && tail) {
      auto tail_epilogue = [&](auto rtag) {
        constexpr int R = decltype(rtag)::value;  // rows per wavefront; this lane: rows R q + sub, group g
        constexpr int G = 32 / R;
        const int sub = lane / G, g = lane % G;
        const float bg = base[(size_t)kt * KT + g];
#pragma unroll
        for (int j = 0; j < RL; j++) {
          const size_t rb = (row0 - row_org) / 32 + j;
          if (row0 + (size_t)j * 32 < row_hi) {
            float *dst = scores + (rb * ld + (size_t)kt * KT + g) * 32 + sub;
#pragma unroll
            for (int q = 0; q < G; q++) dst[q * R] = acc[j * G + q][0] + bg;
          }
        }
      };
      if (tail_g == 8) tail_epilogue(std::integral_constant<int, 4>{});
      else tail_epilogue(std::integral_constant<int, 2>{});
    } else {
      VecF<V> b;
      b.load(base + (size_t)kt * KT + lane * V);
#pragma unroll
      for (int j = 0; j < RL; j++) {
        const size_t rb = (row0 - row_org) / 32 + j;
        if (row0 + (size_t)j * 32 < row_hi) {
#pragma unroll
          for (int v = 0; v < V; v++) {
            float4 *dst = reinterpret_cast<float4 *>(scores + (rb * ld + (size_t)kt * KT + lane * V + v) * 32);
#pragma unroll
            for (int r4 = 0; r4 < 8; r4++)
              dst[r4] = make_float4(acc[j * 32 + r4 * 4 + 0][v] + b.v[v], acc[j * 32 + r4 * 4 + 1][v] + b.v[v],
                                    acc[j * 32 + r4 * 4 + 2][v] + b.v[v], acc[j * 32 + r4 * 4 + 3][v] + b.v[v]);
          }
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// score_bundle_kernel -- the general score kernel (states with nich features, slow-path cells, ...).
//
// Same mapping as score_kernel: a block owns NW*RW rows and one k-tile of 32*V groups, lane l owns V consecutive
// groups, acc[RW][V] lives in registers across all features.  What differs is the stage ring: a stage holds a BUNDLE
// of consecutive features of the walk order (their row values, slow masks and parameter chunks, packed at the
// offsets the host laid out: FeatDev::sx_off / sc_off / bundle_last), and the ring is waited for, released and
// refilled once per bundle instead of once per feature.  ncu on the per-feature ring (profiles/r02_c5_score_src.txt):
// one third of C5's warp samples sat in the loop head and tail -- the try_wait round trip, the FeatS reload, the kind
// dispatch, the release atomic whose return value decides who refills -- because a table feature is only ~170
// instructions of work per warp.  A C5 bundle is one period of the walk order (bb, gp, dd, nich: ~64 KB).
// ---------------------------------------------------------------------------------------------------
template <int V, int RW, int NW, bool BLOCKED>
__global__ void __launch_bounds__(NW * 32, 1)
score_bundle_kernel(const FeatDev *__restrict__ feats, int nfeat, const float *__restrict__ params, size_t region_rows,
                    uint32_t stage_bytes, int S, const float *__restrict__ base, float *__restrict__ scores, size_t ld,
                    size_t row_org, size_t row_lo, size_t row_hi, const double *__restrict__ hp,
                    const double *__restrict__ ss, const int32_t *__restrict__ col2slot, int ncols, int ktiles,
                    int *__restrict__ rowmax) {
  constexpr int KT = 32 * V;
  constexpr int RL = (RW + 31) / 32;                            // slow-mask words per warp (RW = 16: half a word)
  constexpr int RB = NW * RW;                                   // rows per block
  constexpr uint32_t X_BYTES = RB * 4, M_BYTES = RB / 8;        // row values, slow masks
  static_assert((RW % 32 == 0 || RW == 16) && M_BYTES % 16 == 0, "tile sizes must keep the bulk copies 16-byte granular");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // layout: [S stages | full[S], release counters[S] | nb | feature table | bundle starts (nfeat + 1) | bundle bytes (nfeat)]
  unsigned char *stages = smem_raw;
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)S * stage_bytes);
  int *nb_slot = reinterpret_cast<int *>(bars + 2 * S);
  FeatS *ftab = reinterpret_cast<FeatS *>(bars + 2 * S + 1);
  uint16_t *bfirst = reinterpret_cast<uint16_t *>(ftab + nfeat);
  uint32_t *bbytes = reinterpret_cast<uint32_t *>(bfirst + ((nfeat + 1 + 1) & ~1));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int kt = (int)(blockIdx.x % (unsigned)ktiles);          // k-tile fastest: a row tile's values come from DRAM once
  const float *region = params + (size_t)kt * region_rows * KT;
  const size_t blk_row0 = row_org + (size_t)(blockIdx.x / (unsigned)ktiles) * RB;   // multiple of 128
  const size_t row0 = blk_row0 + (size_t)warp * RW;

  for (int i = tid; i < nfeat; i += NW * 32) {
    const FeatDev f = feats[i];
    FeatS t;
    t.scol = f.scol; t.slowmask = f.slowmask; t.col = f.col;
    t.rowoff = f.rowoff; t.rows = f.rows; t.ncat = f.ncat;
    t.kind = (uint16_t)((f.kind == KIND_TABLE && f.binform) ? KIND_BIN : f.kind); t.has_slow = (uint16_t)(f.has_slow != 0);
    t.sx_off = f.sx_off; t.sc_off = f.sc_off; t.last = f.bundle_last; t.fuse = f.fuse;
    ftab[i] = t;
  }
  if (tid == 0) {
    for (int s = 0; s < S; s++) {
      mbar_init(smem_u32(&bars[s]), 1);
      bars[S + s] = 0;  // release counter of the stage
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid == 0) {  // bundle table
    int nb = 0;
    uint32_t bytes = 0;
    bfirst[0] = 0;
    for (int i = 0; i < nfeat; i++) {
      const FeatS t = ftab[i];
      bytes += X_BYTES + (t.has_slow ? M_BYTES : 0u) + t.rows * (uint32_t)(KT * sizeof(float));
      if (t.last || i == nfeat - 1) { bbytes[nb] = bytes; bytes = 0; bfirst[++nb] = (uint16_t)(i + 1); }
    }
    *nb_slot = nb;
  }
  __syncthreads();
  const int nb = *nb_slot;

  // one WARP (all 32 lanes converged): everything bundle b needs -> stage s.  Lane 0 arms the barrier, then every lane
  // issues its share of the bundle's copies (three per feature: row values, slow masks, parameter chunk).  One lane
  // issuing the ~20 bulk copies of a C5 bundle one behind the other was the refill's latency: ncu had every warp waiting
  // ~1200 cycles for the full barrier at every bundle start (8.8 % of the samples) although the refill is requested a
  // whole bundle -- ~13000 cycles -- ahead.
  auto issue = [&](int b, int s) {
    const uint32_t bar = smem_u32(&bars[s]);
    const uint32_t dst0 = smem_u32(stages + (size_t)s * stage_bytes);
    if (lane == 0) mbar_expect_tx(bar, bbytes[b]);
    __syncwarp();
    const int d0 = bfirst[b], nc = 3 * (bfirst[b + 1] - d0);
    for (int c = lane; c < nc; c += 32) {
      const FeatS t = ftab[d0 + c / 3];
      const int which = c % 3;
      if (which == 0) bulk_g2s(dst0 + t.sx_off, t.scol + blk_row0, X_BYTES, bar);
      else if (which == 1) { if (t.has_slow) bulk_g2s(dst0 + t.sx_off + X_BYTES, t.slowmask + (blk_row0 >> 5), M_BYTES, bar); }
      else bulk_g2s(dst0 + t.sc_off, region + (size_t)t.rowoff * KT, t.rows * (uint32_t)(KT * sizeof(float)), bar);
    }
    __syncwarp();
  };
  if (warp == 0)
    for (int b = 0; b < S && b < nb; b++) issue(b, b);

  float acc[RW][V];
#pragma unroll
  for (int r = 0; r < RW; r++)
#pragma unroll
    for (int v = 0; v < V; v++) acc[r][v] = 0.f;

  // ---- rare-path fix-ups, shared by the sequential and the fused walk (static register indexing throughout: acc must
  // not spill to local memory)
  auto load_slow = [&](const FeatS &t, const unsigned char *st, uint32_t (&slow)[RL]) {
    if constexpr (RW == 16) {  // two warps share a 32-row mask word
      const uint32_t w = t.has_slow ? reinterpret_cast<const uint32_t *>(st + X_BYTES)[warp >> 1] : 0u;
      slow[0] = (w >> (16 * (warp & 1))) & 0xFFFFu;
    } else {
#pragma unroll
      for (int j = 0; j < RL; j++)
        slow[j] = t.has_slow ? reinterpret_cast<const uint32_t *>(st + X_BYTES)[warp * RL + j] : 0u;
    }
  };
  // bb in binary form: masked cells were scored as x = 0: take back the t0 that base[] carries for this feature
  auto fix_bin = [&](const float *chunk, const uint32_t (&slow)[RL]) {
#pragma unroll
    for (int j = 0; j < RL; j++) {
      uint32_t m = slow[j];
      if (m) {
        VecF<V> t0;
        t0.load(chunk + 1 * KT);
        while (m) {
          const int rr = j * 32 + __ffs(m) - 1;
          m &= m - 1;
#pragma unroll
          for (int r = 0; r < RW; r++)
            if (r == rr)
#pragma unroll
              for (int v = 0; v < V; v++) acc[r][v] -= t0.v[v];
        }
      }
    }
  };
  // gp / bnb counts beyond the table: the fp64 closed form from the suffstats
  auto fix_gp = [&](const FeatS &t, int d, const uint32_t (&slow)[RL]) {
    const uint32_t *raw = reinterpret_cast<const uint32_t *>(t.col);
#pragma unroll
    for (int j = 0; j < RL; j++) {
      uint32_t m = slow[j];
      while (m) {
        const int rr = j * 32 + __ffs(m) - 1;
        m &= m - 1;
        const double xv = (double)raw[row0 + rr];
        float add[V];
#pragma unroll
        for (int v = 0; v < V; v++) {
          const int col = kt * KT + lane * V + v;
          add[v] = 0.f;
          if (col < ncols) add[v] = gp_overflow_score(feats + d, hp, ss, col2slot[col], xv);
        }
#pragma unroll
        for (int r = 0; r < RW; r++)
          if (r == rr)
#pragma unroll
            for (int v = 0; v < V; v++) acc[r][v] += add[v];
      }
    }
  };
  // nich: masked cells were scored as x = 0: undo that term and the c0 that base[] carries for this feature
  auto fix_nich = [&](const float *chunk, const VecF<V> &mu, const VecF<V> &sc, const VecF<V> &c1, const uint32_t (&slow)[RL]) {
#pragma unroll
    for (int j = 0; j < RL; j++) {
      uint32_t m = slow[j];
      if (m) {
        VecF<V> c0;
        c0.load(chunk + 3 * KT);
        float undo[V];
#pragma unroll
        for (int v = 0; v < V; v++) {
          const float tt = (0.f - mu.v[v]) * sc.v[v];
          undo[v] = -fmaf(c1.v[v], log2_1p_pos(tt * tt), c0.v[v]);
        }
        while (m) {
          const int rr = j * 32 + __ffs(m) - 1;
          m &= m - 1;
#pragma unroll
          for (int r = 0; r < RW; r++)
            if (r == rr)
#pragma unroll
              for (int v = 0; v < V; v++) acc[r][v] += undo[v];
        }
      }
    }
  };

  int s = 0;
  uint32_t parity = 0;
  for (int b = 0; b < nb; b++) {
    mbar_wait(smem_u32(&bars[s]), parity);
    const unsigned char *stage = stages + (size_t)s * stage_bytes;
    const int d1 = bfirst[b + 1];
    for (int d = bfirst[b]; d < d1; d++) {
      const FeatS t = ftab[d];
      const unsigned char *st = stage + t.sx_off;
      // this warp's RW row values, read as broadcast 128-bit loads (4 rows per shared-memory wavefront)
      const uint4 *xq = reinterpret_cast<const uint4 *>(st) + warp * (RW / 4);
      const float *chunk = reinterpret_cast<const float *>(stage + t.sc_off) + lane * V;
      uint32_t slow[RL];
      load_slow(t, st, slow);

      if constexpr (V == 4) {
        if (t.fuse) {
          // Fused quad [bb in binary form, table A, table B, nich] (the host orders the walk so; all four sit in this
          // stage): every row step issues the two lookups (shared-memory pipe) next to the nich arithmetic (FMA / XU
          // pipes) and the bb multiply-add, so that inside ONE warp the lookup latency hides under ~30 arithmetic
          // instructions and both pipes stay busy.  Walking the four features one after the other keeps each pipe idle
          // while the other works: with 242 registers there are only two warps per scheduler to overlap anything.
          const FeatS tA = ftab[d + 1], tC = ftab[d + 2], tN = ftab[d + 3];
          const unsigned char *stA = stage + tA.sx_off, *stC = stage + tC.sx_off, *stN = stage + tN.sx_off;
          const uint4 *xqA = reinterpret_cast<const uint4 *>(stA) + warp * (RW / 4);
          const uint4 *xqC = reinterpret_cast<const uint4 *>(stC) + warp * (RW / 4);
          const uint4 *xqN = reinterpret_cast<const uint4 *>(stN) + warp * (RW / 4);
          const float *chunkA = reinterpret_cast<const float *>(stage + tA.sc_off) + lane * V;
          const float *chunkC = reinterpret_cast<const float *>(stage + tC.sc_off) + lane * V;
          const float *chunkN = reinterpret_cast<const float *>(stage + tN.sc_off) + lane * V;
          const uint32_t cA = smem_u32(chunkA), cC = smem_u32(chunkC);
          VecF<V> df, mu, sc, c1;
          df.load(chunk + 0 * KT);
          mu.load(chunkN + 0 * KT);
          sc.load(chunkN + 1 * KT);
          c1.load(chunkN + 2 * KT);
          float2 nmu2[2], sc2[2], c12[2], df2[2];
#pragma unroll
          for (int h = 0; h < 2; h++) {
            nmu2[h] = make_float2(-mu.v[2 * h], -mu.v[2 * h + 1]);
            sc2[h] = make_float2(sc.v[2 * h], sc.v[2 * h + 1]);
            c12[h] = make_float2(c1.v[2 * h], c1.v[2 * h + 1]);
            df2[h] = make_float2(df.v[2 * h], df.v[2 * h + 1]);
          }
#pragma unroll
          for (int r4 = 0; r4 < RW / 4; r4++) {
            const uint4 qB = xq[r4], qA = xqA[r4], qC = xqC[r4], qN = xqN[r4];
            const float xb[4] = {__uint_as_float(qB.x), __uint_as_float(qB.y), __uint_as_float(qB.z), __uint_as_float(qB.w)};
            const float xn[4] = {__uint_as_float(qN.x), __uint_as_float(qN.y), __uint_as_float(qN.z), __uint_as_float(qN.w)};
            const uint32_t iA[4] = {qA.x, qA.y, qA.z, qA.w}, iC[4] = {qC.x, qC.y, qC.z, qC.w};
#pragma unroll
            for (int e = 0; e < 4; e++) {
              const int r = r4 * 4 + e;
              VecF<V> tvA, tvC;
              lds_vec<V>(tvA.v, cA + iA[e] * (uint32_t)(KT * sizeof(float)));
              lds_vec<V>(tvC.v, cC + iC[e] * (uint32_t)(KT * sizeof(float)));
              const float2 x2 = make_float2(xn[e], xn[e]), b2 = make_float2(xb[e], xb[e]);
#pragma unroll
              for (int h = 0; h < 2; h++) {
                const float2 tt = __fmul2_rn(__fadd2_rn(x2, nmu2[h]), sc2[h]);
                float2 a = __ffma2_rn(c12[h], log2_1p_pos2(__fmul2_rn(tt, tt)), make_float2(acc[r][2 * h], acc[r][2 * h + 1]));
                a = __ffma2_rn(b2, df2[h], a);
                a = __fadd2_rn(a, make_float2(tvA.v[2 * h], tvA.v[2 * h + 1]));
                a = __fadd2_rn(a, make_float2(tvC.v[2 * h], tvC.v[2 * h + 1]));
                acc[r][2 * h] = a.x;
                acc[r][2 * h + 1] = a.y;
              }
            }
          }
          // rare paths of the four features
          fix_bin(chunk, slow);
          uint32_t slowX[RL];
          if (tA.kind == KIND_GP) { load_slow(tA, stA, slowX); fix_gp(tA, d + 1, slowX); }
          if (tC.kind == KIND_GP) { load_slow(tC, stC, slowX); fix_gp(tC, d + 2, slowX); }
          load_slow(tN, stN, slowX);
          fix_nich(chunkN, mu, sc, c1, slowX);
          d += 3;
          continue;
        }
      }

      if (t.kind == KIND_BIN) {  // bb in binary form: acc += x (t1 - t0), sum_d t0 is already in base[]
        VecF<V> df;
        df.load(chunk + 0 * KT);
#pragma unroll
        for (int r4 = 0; r4 < RW / 4; r4++) {
          const uint4 q = xq[r4];
          const float xs[4] = {__uint_as_float(q.x), __uint_as_float(q.y), __uint_as_float(q.z), __uint_as_float(q.w)};
#pragma unroll
          for (int e = 0; e < 4; e++) {
            if constexpr (V % 2 == 0) {
#pragma unroll
              for (int h = 0; h < V / 2; h++) {
                const float2 a = __ffma2_rn(make_float2(xs[e], xs[e]), make_float2(df.v[2 * h], df.v[2 * h + 1]),
                                            make_float2(acc[r4 * 4 + e][2 * h], acc[r4 * 4 + e][2 * h + 1]));
                acc[r4 * 4 + e][2 * h] = a.x;
                acc[r4 * 4 + e][2 * h + 1] = a.y;
              }
            } else {
#pragma unroll
              for (int v = 0; v < V; v++) acc[r4 * 4 + e][v] = fmaf(xs[e], df.v[v], acc[r4 * 4 + e][v]);
            }
          }
        }
        fix_bin(chunk, slow);
      } else if (t.kind != KIND_NICH) {
        const uint32_t chunk_s = smem_u32(chunk);
#pragma unroll
        for (int r4 = 0; r4 < RW / 4; r4++) {
          const uint4 q = xq[r4];
          const uint32_t idx[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
          for (int e = 0; e < 4; e++) {
            VecF<V> tv;
            lds_vec<V>(tv.v, chunk_s + idx[e] * (uint32_t)(KT * sizeof(float)));
            if constexpr (V % 2 == 0) {
#pragma unroll
              for (int h = 0; h < V / 2; h++) {
                const float2 a = __fadd2_rn(make_float2(acc[r4 * 4 + e][2 * h], acc[r4 * 4 + e][2 * h + 1]),
                                            make_float2(tv.v[2 * h], tv.v[2 * h + 1]));
                acc[r4 * 4 + e][2 * h] = a.x;
                acc[r4 * 4 + e][2 * h + 1] = a.y;
              }
            } else {
#pragma unroll
              for (int v = 0; v < V; v++) acc[r4 * 4 + e][v] += tv.v[v];
            }
          }
        }
        if (t.kind == KIND_GP) fix_gp(t, d, slow);
      } else {  // KIND_NICH: c1' log2(1 + ((x - mu) s)^2); sum_d c0 is already in base[]
        VecF<V> mu, sc, c1;
        mu.load(chunk + 0 * KT);
        sc.load(chunk + 1 * KT);
        c1.load(chunk + 2 * KT);
        if constexpr (V % 2 == 0) {  // two groups per instruction (FADD2 / FMUL2 / FFMA2)
          float2 nmu2[V / 2], sc2[V / 2], c12[V / 2];
#pragma unroll
          for (int h = 0; h < V / 2; h++) {
            nmu2[h] = make_float2(-mu.v[2 * h], -mu.v[2 * h + 1]);
            sc2[h] = make_float2(sc.v[2 * h], sc.v[2 * h + 1]);
            c12[h] = make_float2(c1.v[2 * h], c1.v[2 * h + 1]);
          }
#pragma unroll
          for (int r4 = 0; r4 < RW / 4; r4++) {
            const uint4 q = xq[r4];
            const float xs[4] = {__uint_as_float(q.x), __uint_as_float(q.y), __uint_as_float(q.z), __uint_as_float(q.w)};
#pragma unroll
            for (int e = 0; e < 4; e++) {
              const float2 x2 = make_float2(xs[e], xs[e]);
#pragma unroll
              for (int h = 0; h < V / 2; h++) {
                const float2 tt = __fmul2_rn(__fadd2_rn(x2, nmu2[h]), sc2[h]);
                const float2 a = __ffma2_rn(c12[h], log2_1p_pos2(__fmul2_rn(tt, tt)),
                                            make_float2(acc[r4 * 4 + e][2 * h], acc[r4 * 4 + e][2 * h + 1]));
                acc[r4 * 4 + e][2 * h] = a.x;
                acc[r4 * 4 + e][2 * h + 1] = a.y;
              }
            }
          }
        } else {
#pragma unroll
          for (int r4 = 0; r4 < RW / 4; r4++) {
            const uint4 q = xq[r4];
            const float xs[4] = {__uint_as_float(q.x), __uint_as_float(q.y), __uint_as_float(q.z), __uint_as_float(q.w)};
#pragma unroll
            for (int e = 0; e < 4; e++)
#pragma unroll
              for (int v = 0; v < V; v++) {
                const float tt = (xs[e] - mu.v[v]) * sc.v[v];
                acc[r4 * 4 + e][v] = fmaf(c1.v[v], log2_1p_pos(tt * tt), acc[r4 * 4 + e][v]);
              }
          }
        }
        fix_nich(chunk, mu, sc, c1, slow);
      }
    }
    // Release the stage: a counter per stage, and the warp that arrives LAST issues the refill with bundle b + S, so
    // that nobody waits here (see score_kernel for what was measured against a fixed producer thread).
    __syncwarp();
    unsigned int last = 0;
    if (lane == 0) {
      const uint32_t rel = smem_u32(&bars[S + s]);
      unsigned int old;
      asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(rel) : "memory");
      if (old == (unsigned)(NW - 1)) {
        asm volatile("st.relaxed.cta.shared::cta.u32 [%0], %1;" ::"r"(rel), "r"(0u) : "memory");
        last = 1;
      }
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (last && b + S < nb) issue(b + S, s);   // the whole warp issues (see issue)
    if (++s == S) { s = 0; parity ^= 1u; }
  }

  // epilogue: + log(pseudocount) (group_manager.hpp:274-283)
  VecF<V> bv;
  bv.load(base + (size_t)kt * KT + lane * V);
  if constexpr (!BLOCKED) {  // 128 V-byte coalesced row-major stores
#pragma unroll
    for (int r = 0; r < RW; r++) {
      const size_t row = row0 + r;
      if (row >= row_lo && row < row_hi) {
        float o[V];
#pragma unroll
        for (int v = 0; v < V; v++) o[v] = acc[r][v] + bv.v[v];
        store_vec<V>(scores + (row - row_org) * ld + (size_t)kt * KT + lane * V, o);
      }
    }
  } else {
    // transpose each 32-row x KT-group tile through shared memory (the drained stage ring) so that
    // lane = row and every store instruction writes 32 consecutive floats of one group
    __syncthreads();  // every warp has finished reading the stages
    if constexpr (RW == 16) {  // a pair of warps owns one 32-row block: each writes its 16 rows, each stores half of the columns
      float *tile = reinterpret_cast<float *>(stages) + (size_t)(warp >> 1) * 32 * (KT + 1);
      const int rbase = 16 * (warp & 1);
#pragma unroll
      for (int r = 0; r < 16; r++)
#pragma unroll
        for (int v = 0; v < V; v++) tile[(rbase + r) * (KT + 1) + lane * V + v] = acc[r][v] + bv.v[v];
      __syncthreads();
      const size_t prow0 = blk_row0 + (size_t)(warp >> 1) * 32;
      if (prow0 < row_hi) {
        float *dst = scores + (((prow0 - row_org) / 32) * ld + (size_t)kt * KT) * 32 + lane;
        const int c0 = (warp & 1) * (KT / 2);
        float mx = -CUDART_INF_F;
#pragma unroll 8
        for (int c = c0; c < c0 + KT / 2; c++) {
          const float v = tile[lane * (KT + 1) + c];
          dst[(size_t)c * 32] = v;
          if (kt * KT + c < ncols) mx = fmaxf(mx, v);
        }
        if (rowmax) atomicMax(rowmax + (prow0 - row_org) + lane, float_ordered(mx));
      }
      return;
    }
    float *tile = reinterpret_cast<float *>(stages) + (size_t)warp * 32 * (KT + 1);
#pragma unroll
    for (int j = 0; j < RL; j++) {
      __syncwarp();
#pragma unroll
      for (int r = 0; r < 32; r++)
#pragma unroll
        for (int v = 0; v < V; v++) tile[r * (KT + 1) + lane * V + v] = acc[j * 32 + r][v] + bv.v[v];
      __syncwarp();
      const size_t rb = (row0 - row_org) / 32 + j;
      if (row0 + (size_t)j * 32 < row_hi) {
        float *dst = scores + (rb * ld + (size_t)kt * KT) * 32 + lane;
        // the row's largest score over this k-tile's real groups goes to the sampler (atomic max over the k-tiles of
        // the row, floats ordered as integers): its first pass over the score matrix -- the maximum -- is then not needed
        float mx = -CUDART_INF_F;
#pragma unroll 8
        for (int c = 0; c < KT; c++) {
          const float v = tile[lane * (KT + 1) + c];
          dst[(size_t)c * 32] = v;
          if (kt * KT + c < ncols) mx = fmaxf(mx, v);
        }
        if (rowmax) atomicMax(rowmax + rb * 32 + lane, float_ordered(mx));
      }
    }
  }
}

}  // namespace msb
