// msb_kernels.cuh -- sm_100a kernels of the hot path (see DESIGN.md for the
// data layout, the per-kernel roofline and the algorithmic bytes).
#pragma once
#include <cstddef>
#include <string>
#include <vector>

#include "msb_math.cuh"

namespace msb {

// Optional per-kernel timing (msb_ctx_profile): a CUDA event pair around every launch while it is switched on.
// Off by default -- nothing is recorded on the hot path.  Used by bench.py for one extra, untimed step so that the
// bandwidth-bound kernels (ingest, sampler, update, conversions) can each be reported against the HBM roof.
struct KernelProf {
  struct Rec { const char *name; cudaEvent_t a, b; };
  bool on = false;
  cudaStream_t stream = nullptr;
  std::vector<Rec> recs;
  std::vector<cudaEvent_t> pool;
  cudaEvent_t take() {
    cudaEvent_t e = nullptr;
    if (!pool.empty()) { e = pool.back(); pool.pop_back(); }
    else cudaEventCreate(&e);
    return e;
  }
  void begin(const char *name, cudaStream_t s) {
    if (!on) return;
    Rec r{name, take(), take()};
    cudaEventRecord(r.a, s);
    recs.push_back(r);
  }
  void end(cudaStream_t s) {
    if (!on || recs.empty()) return;
    cudaEventRecord(recs.back().b, s);
  }
  void clear() {
    for (auto &r : recs) { pool.push_back(r.a); pool.push_back(r.b); }
    recs.clear();
  }
  void destroy() {
    clear();
    for (auto e : pool) cudaEventDestroy(e);
    pool.clear();
  }
};

enum Kind : int { KIND_TABLE = 0, KIND_GP = 1, KIND_NICH = 2, KIND_NIW = 3, KIND_DM = 4,
                  KIND_BIN = 5 };  // KIND_BIN: score-kernel-local code of a KIND_TABLE feature in binary form (FeatDev::binform)
enum ColType : int { COL_U8 = 0, COL_U16 = 1, COL_U32 = 2, COL_F32 = 3 };

constexpr uint32_t GP_SENTINEL = 0xFFFFFFFFu;

// Per-feature descriptor, one array in device memory per state.
struct FeatDev {
  int32_t family;     // Family
  int32_t kind;       // Kind
  int32_t coltype;    // ColType
  uint32_t dim;       // dd categories / niw dimension / bb 2
  uint32_t ncat;      // table categories: bb 2, dd dim, gp cap; index ncat = zero row (masked)
  uint32_t rows;      // rows of this feature's parameter chunk (each row = KT floats)
  uint32_t rowoff;    // first row of the chunk inside a k-tile region
  uint32_t ss_w;      // doubles per group slot
  const void *col;    // Value-typed column, n elements (niw: n x dim floats)
  const uint32_t *scol;     // score column: u32 table row index (always a valid chunk row) or f32 value (masked -> 0);
                            // niw: the CENTRED rows, f32[n][dim] = x - c (what the fp32 scorers read; col keeps the raw rows)
  const uint32_t *slowmask; // per 32-row block: rows that need the score kernel's slow path (gp overflow, nich masked);
                            // niw: the centre c, f32[dim] (0 for coordinates that are not far from the origin)
  uint32_t has_slow;        // any bit set in slowmask
  uint32_t binform;         // bb next to nich features: scored as base + x * (t1 - t0) on the FMA pipe instead of a table lookup
                            // (chunk rows: t1 - t0, t0; score column: x as 0.0f / 1.0f, masked cells 0 with their slow bit set)
  uint64_t hp_off;    // into hp[]
  uint64_t ss_off;    // into ss[] / delta[]: block[slot * ss_w + j]
  double asum;        // dd: sum of alphas.  nich: the centre c of the score column (x' = x - c; 0 unless the whole column is far from 0)
  // AoS source record (row_major_dataview layout, runtime_type.hpp:123-134)
  uint64_t src_off;
  uint64_t msk_off;
  uint32_t src_prim;
  uint32_t src_n;
  // score_bundle_kernel: where the feature sits inside the shared-memory stage of its bundle (laid out by the host for
  // the tile shape in use), and whether it closes the bundle
  uint32_t sx_off;
  uint32_t sc_off;
  uint32_t bundle_last;
  uint32_t fuse;      // first feature of a fused quad [bb in binary form, table, table, nich] (all four in one bundle)
};

__device__ __forceinline__ void atomic_add_f64(double *p, double v) { atomicAdd(p, v); }

// ---------------------------------------------------------------------------
// AoS -> SoA pack: applies runtime_cast (runtime_type.hpp:145-166) once per
// cell and folds the mask in-band (sentinel value per column type).
// ---------------------------------------------------------------------------
__device__ __forceinline__ double load_prim(const uint8_t *p, uint32_t prim) {
  switch (prim) {
    case 0: return (double)(*p != 0);
    case 1: return (double)*(const int8_t *)p;
    case 2: return (double)*p;
    case 3: { int16_t v; memcpy(&v, p, 2); return (double)v; }
    case 4: { uint16_t v; memcpy(&v, p, 2); return (double)v; }
    case 5: { int32_t v; memcpy(&v, p, 4); return (double)v; }
    case 6: { uint32_t v; memcpy(&v, p, 4); return (double)v; }
    case 7: { long long v; memcpy(&v, p, 8); return (double)v; }
    case 8: { unsigned long long v; memcpy(&v, p, 8); return (double)v; }
    case 9: { float v; memcpy(&v, p, 4); return (double)v; }
    default: { double v; memcpy(&v, p, 8); return v; }
  }
}
__device__ __forceinline__ uint32_t prim_size(uint32_t prim) {
  // sizes {1, 1, 1, 2, 2, 4, 4, 8, 8, 4, 8} of type_info.h:10-34 as nibbles of one constant (an indexed local array costs every
  // thread eleven local-memory stores per call: 4 % of the ingest kernel's instructions in the round-2 profile)
  return (uint32_t)((0x84884422111ull >> (4u * prim)) & 0xFull);
}

__global__ void pack_kernel(const uint8_t *__restrict__ data, const uint8_t *__restrict__ mask, size_t n,
                            size_t rowsize, size_t maskrowsize, const FeatDev *__restrict__ feats, int nfeat) {
  const size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int d = blockIdx.y;
  if (row >= n || d >= nfeat) return;
  const FeatDev f = feats[d];
  const uint8_t *src = data + row * rowsize + f.src_off;
  bool masked = false;
  if (mask) {
    const uint8_t *m = mask + row * maskrowsize + f.msk_off;
    for (uint32_t i = 0; i < f.src_n; i++) masked |= (m[i] != 0);
  }
  const uint32_t ps = prim_size(f.src_prim);
  if (f.kind == KIND_NIW) {
    float *dst = (float *)f.col + row * (size_t)f.dim;
    for (uint32_t i = 0; i < f.dim; i++) dst[i] = (float)load_prim(src + i * ps, f.src_prim);
    if (masked) dst[0] = CUDART_NAN_F;
    return;
  }
  if (f.kind == KIND_DM) {  // a row of dim counts; masked row: sentinel in element 0
    uint32_t *dst = (uint32_t *)f.col + row * (size_t)f.dim;
    for (uint32_t i = 0; i < f.dim; i++) {
      const double c = load_prim(src + i * ps, f.src_prim);
      dst[i] = c < 0.0 ? 0u : (c >= 4294967294.0 ? 4294967294u : (uint32_t)c);
    }
    if (masked) dst[0] = GP_SENTINEL;
    return;
  }
  const double v = load_prim(src, f.src_prim);
  if (f.kind == KIND_NICH) {
    ((float *)f.col)[row] = masked ? CUDART_NAN_F : (float)v;
  } else if (f.kind == KIND_GP) {
    uint32_t x = v < 0.0 ? 0u : (v >= 4294967294.0 ? 4294967294u : (uint32_t)v);
    ((uint32_t *)f.col)[row] = masked ? GP_SENTINEL : x;
  } else {  // bb / dd category; out-of-range categories are treated as masked
    uint32_t x = f.ncat;
    if (!masked) {
      if (f.family == FAM_BB) x = (v != 0.0) ? 1u : 0u;
      else if (v >= 0.0 && v < (double)f.ncat) x = (uint32_t)v;
    }
    if (f.coltype == COL_U8) ((uint8_t *)f.col)[row] = (uint8_t)x;
    else if (f.coltype == COL_U16) ((uint16_t *)f.col)[row] = (uint16_t)x;
    else ((uint32_t *)f.col)[row] = x;
  }
}

// Score columns: what the score kernel streams.  One u32 per (row, feature): the chunk row to look up
// (masked cells and gp counts beyond the table point at the all-zero row) or the f32 value (masked -> 0),
// plus a bitmask per 32-row block of the cells that need the slow path.  Rows [n, n_pad) are padding.
__global__ void scorecol_kernel(const FeatDev *__restrict__ feats, int nfeat, size_t n, size_t n_pad,
                                uint32_t *__restrict__ any_slow) {
  const size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // n_pad is a multiple of the block size
  const int d = blockIdx.y;
  const FeatDev f = feats[d];
  if (f.kind == KIND_NIW || f.kind == KIND_DM) return;
  uint32_t out;
  bool slow = false;
  if (f.kind == KIND_NICH) {
    const float x = row < n ? ((const float *)f.col)[row] : 0.f;
    slow = x != x;
    out = (slow || row >= n) ? 0u : __float_as_uint((float)((double)x - f.asum));  // centred, see build_params_kernel
  } else if (f.kind == KIND_GP) {
    const uint32_t x = row < n ? ((const uint32_t *)f.col)[row] : GP_SENTINEL;
    slow = x != GP_SENTINEL && x >= f.ncat;
    out = x < f.ncat ? x : f.ncat;
  } else {
    uint32_t x = f.ncat;
    if (row < n) {
      if (f.coltype == COL_U8) x = ((const uint8_t *)f.col)[row];
      else if (f.coltype == COL_U16) x = ((const uint16_t *)f.col)[row];
      else x = ((const uint32_t *)f.col)[row];
    }
    out = x < f.ncat ? x : f.ncat;
    if (f.binform) {  // binary form: the value itself; masked / out-of-range cells take the slow path
      slow = row < n && x >= f.ncat;
      out = __float_as_uint(x == 1u ? 1.0f : 0.0f);
    }
  }
  const_cast<uint32_t *>(f.scol)[row] = out;
  const uint32_t m = __ballot_sync(0xffffffffu, slow);
  if ((threadIdx.x & 31) == 0) {
    const_cast<uint32_t *>(f.slowmask)[row >> 5] = m;
    if (m) any_slow[d] = 1u;
  }
}

// pack_kernel + scorecol_kernel in one pass with the AoS records staged in shared memory: a block copies TR
// consecutive records (and their mask rows) with coalesced 4-byte loads into a padded tile (pitch = record
// words + 1: thread = row reads of one field are bank-conflict free), then thread r converts every field of
// row r and writes the Value-typed column, the score column and (by ballot) the slow-path mask.  The records
// are read from HBM exactly once.  Needs the gp table sizes (refresh path; bind sizes them first).
// rowsize and maskrowsize are multiples of 4 here (the host falls back to the two-kernel path otherwise).
// NS slices of TR threads each: thread (r, slice) converts the features d = slice, slice + NS, ... of row r, so a warp is
// still 32 consecutive rows of one feature (coalesced column stores, one ballot per slow-path word) and a block keeps
// NS * TR / 32 = 16 warps busy whatever the record size (round 1: one thread per row walked all D features -- 2 warps per
// scheduler, 7 % of the HBM roof on C5).  TR is chosen by the host so that several blocks fit in an SM's shared memory and
// one block's tile load overlaps another's conversion.  The per-feature descriptors are read from global memory
// (warp-uniform, L1-resident).
template <int TR, int NS>
__global__ void __launch_bounds__(TR * NS)
ingest_tile_kernel(const uint8_t *__restrict__ data, const uint8_t *__restrict__ mask, size_t n, size_t n_pad,
                   uint32_t rowwords, uint32_t maskwords, const FeatDev *__restrict__ feats, int nfeat,
                   uint32_t *__restrict__ any_slow) {
  extern __shared__ uint32_t tile[];
  constexpr int NT = TR * NS;
  const uint32_t pitch = rowwords + 1, mpitch = maskwords + 1;
  uint32_t *mtile = tile + (size_t)TR * pitch;
  const size_t row0 = (size_t)blockIdx.x * TR;
  const size_t rows_here = row0 < n ? min((size_t)TR, n - row0) : 0;
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(data) + row0 * rowwords;
    const uint32_t total = (uint32_t)rows_here * rowwords;
    if ((rowwords & 3u) == 0 && ((reinterpret_cast<uintptr_t>(src) & 15u) == 0)) {  // 16-byte loads, 4-byte padded stores
      const uint4 *src4 = reinterpret_cast<const uint4 *>(src);
      for (uint32_t g = threadIdx.x; g < total / 4; g += NT) {
        const uint4 v = __ldg(src4 + g);
        const uint32_t w = g * 4, r = w / rowwords, c = w - r * rowwords;
        uint32_t *dst = tile + r * pitch + c;
        dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
      }
    } else {
      for (uint32_t g = threadIdx.x; g < total; g += NT) tile[(g / rowwords) * pitch + g % rowwords] = src[g];
    }
    if (mask) {
      const uint32_t *msrc = reinterpret_cast<const uint32_t *>(mask) + row0 * maskwords;
      const uint32_t mtotal = (uint32_t)rows_here * maskwords;
      for (uint32_t g = threadIdx.x; g < mtotal; g += NT) mtile[(g / maskwords) * mpitch + g % maskwords] = msrc[g];
    }
  }
  __syncthreads();
  const int r = threadIdx.x % TR, slice = threadIdx.x / TR;
  const size_t row = row0 + r;   // n_pad is a multiple of TR: every thread owns a (possibly padding) row
  const bool live = row < n;
  const uint8_t *rec = reinterpret_cast<const uint8_t *>(tile + (size_t)r * pitch);
  const uint8_t *mrec = reinterpret_cast<const uint8_t *>(mtile + (size_t)r * mpitch);
  static_assert(sizeof(FeatDev) % 16 == 0 && offsetof(FeatDev, sx_off) == 112, "the descriptor is fetched as seven 16-byte loads");
  for (int d = slice; d < nfeat; d += NS) {
    // the descriptor (warp-uniform, L1-resident) in seven independent 16-byte loads: one wait per feature instead of one
    // per field (the field-by-field form spent half of the kernel's warp samples on those dependent loads)
    FeatDev f;
    {
      const uint4 *src = reinterpret_cast<const uint4 *>(feats + d);
      uint4 *dst = reinterpret_cast<uint4 *>(&f);
#pragma unroll
      for (int i = 0; i < 7; i++) dst[i] = __ldg(src + i);
    }
    bool masked = false;
    if (mask && live)
      for (uint32_t i = 0; i < f.src_n; i++) masked |= (mrec[f.msk_off + i] != 0);
    const uint32_t ps = prim_size(f.src_prim);
    if (f.kind == KIND_NIW) {
      if (live) {
        float *dst = (float *)f.col + row * (size_t)f.dim;
        float *dsc = (float *)f.scol + row * (size_t)f.dim;
        const float *cen = (const float *)f.slowmask;
        for (uint32_t i = 0; i < f.dim; i++) {
          const double v = load_prim(rec + f.src_off + i * ps, f.src_prim);
          dst[i] = (float)v;
          dsc[i] = (float)((double)(float)v - (double)cen[i]);
        }
        if (masked) dst[0] = dsc[0] = CUDART_NAN_F;
      }
      continue;
    }
    if (f.kind == KIND_DM) {
      if (live) {
        uint32_t *dst = (uint32_t *)f.col + row * (size_t)f.dim;
        for (uint32_t i = 0; i < f.dim; i++) {
          const double c = load_prim(rec + f.src_off + i * ps, f.src_prim);
          dst[i] = c < 0.0 ? 0u : (c >= 4294967294.0 ? 4294967294u : (uint32_t)c);
        }
        if (masked) dst[0] = GP_SENTINEL;
      }
      continue;
    }
    uint32_t out;
    bool slow = false;
    const uint8_t *p = rec + f.src_off;
    // 4-byte sources at 4-byte offsets (the usual record): one aligned shared-memory load instead of four byte loads
    const bool word = (f.src_off & 3u) == 0;
    const uint32_t w32 = word ? *reinterpret_cast<const uint32_t *>(p) : 0u;
    if (f.kind == KIND_NICH) {
      // the cast of runtime_type.hpp:145-166 to the model's float Value: exact for a float source, through double otherwise
      float x;
      if (f.src_prim == 9) { if (word) x = __uint_as_float(w32); else memcpy(&x, p, 4); }
      else x = (float)load_prim(p, f.src_prim);
      if (masked) x = CUDART_NAN_F;
      if (live) ((float *)f.col)[row] = x;
      slow = live && masked;
      out = (slow || !live) ? 0u : __float_as_uint((float)((double)x - f.asum));
    } else {
      // unsigned integer Values (bool, category, count): the common integer sources convert without a trip through double;
      // `big` marks values no uint32 Value holds (they saturate like the double path), `neg` negative sources
      uint32_t xi = 0;
      bool neg = false, big = false;
      switch (f.src_prim) {
        case 0: xi = (*p != 0); break;
        case 2: xi = *p; break;
        case 4: { uint16_t v; memcpy(&v, p, 2); xi = v; break; }
        case 6: if (word) xi = w32; else memcpy(&xi, p, 4); break;
        case 1: { const int8_t v = *(const int8_t *)p; neg = v < 0; xi = (uint32_t)v; break; }
        case 3: { int16_t v; memcpy(&v, p, 2); neg = v < 0; xi = (uint32_t)v; break; }
        case 5: { int32_t v; if (word) v = (int32_t)w32; else memcpy(&v, p, 4); neg = v < 0; xi = (uint32_t)v; break; }
        default: {
          const double v = live ? load_prim(p, f.src_prim) : 0.0;
          neg = v < 0.0; big = v >= 4294967294.0;
          xi = (neg || big) ? 0u : (uint32_t)v;
          if (f.kind != KIND_GP && f.family == FAM_BB) xi = (v != 0.0) ? 1u : 0u, neg = big = false;   // any non-zero value is "true"
          else if (f.kind != KIND_GP && !neg && !big && !(v < (double)f.ncat)) big = true;                // includes fractions >= ncat, NaN
          break;
        }
      }
      if (f.kind == KIND_GP) {
        uint32_t x = neg ? 0u : (big || xi >= 4294967294u ? 4294967294u : xi);
        if (masked || !live) x = GP_SENTINEL;
        if (live) ((uint32_t *)f.col)[row] = x;
        slow = x != GP_SENTINEL && x >= f.ncat;
        out = x < f.ncat ? x : f.ncat;
      } else {
        uint32_t x = f.ncat;
        if (live && !masked) {
          if (f.family == FAM_BB) x = (xi != 0u || neg) ? 1u : 0u;
          else if (!neg && !big && xi < f.ncat) x = xi;
        }
        if (live) {
          if (f.coltype == COL_U8) ((uint8_t *)f.col)[row] = (uint8_t)x;
          else if (f.coltype == COL_U16) ((uint16_t *)f.col)[row] = (uint16_t)x;
          else ((uint32_t *)f.col)[row] = x;
        }
        out = x;
        if (f.binform) {
          slow = live && x >= f.ncat;
          out = __float_as_uint(x == 1u ? 1.0f : 0.0f);
        }
      }
    }
    if (row < n_pad) const_cast<uint32_t *>(f.scol)[row] = out;
    const uint32_t m = __ballot_sync(0xffffffffu, slow);
    if ((threadIdx.x & 31) == 0 && row < n_pad) {
      const_cast<uint32_t *>(f.slowmask)[row >> 5] = m;
      if (m) any_slow[d] = 1u;
    }
  }
}

// per-coordinate sum / count / min / max of a niw column (rows with a NaN first element are masked);
// blockIdx.y = coordinate.  out[j] = [sum, count], minmax[j] = [min key, max key]
__global__ void niw_colstats_kernel(const float *__restrict__ X, size_t n, int d, double *out, uint32_t *minmax) {
  const int j = blockIdx.y;
  double s = 0.0, c = 0.0;
  uint32_t lo = 0xFFFFFFFFu, hi = 0u;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float v = X[i * d + j];
    if (X[i * d] == X[i * d] && v == v) {
      s += (double)v; c += 1.0;
      const uint32_t b = __float_as_uint(v), k = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
      lo = min(lo, k); hi = max(hi, k);
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o); c += __shfl_xor_sync(0xffffffffu, c, o);
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o)); hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out + 2 * j, s); atomicAdd(out + 2 * j + 1, c); atomicMin(minmax + 2 * j, lo); atomicMax(minmax + 2 * j + 1, hi); }
}
// xc = x - c, the masked-row marker (NaN in element 0) kept
__global__ void niw_center_kernel(const float *__restrict__ X, size_t n, int d, const float *__restrict__ cen, float *__restrict__ Xc) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * (size_t)d) return;
  const int j = (int)(i % d);
  const float v = X[i];
  Xc[i] = (j == 0 && v != v) ? v : (float)((double)v - (double)cen[j]);
}

// sum, count, min and max of a nich column (ignoring masked cells): decides the centre of the score column.
// out = [sum, count] as doubles, then [min, max] kept as order-preserving uint32 keys of the floats
__device__ __forceinline__ uint32_t f32_key(float v) { const uint32_t b = __float_as_uint(v); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }
__global__ void colstats_f32_kernel(const float *__restrict__ col, size_t n, double *out, uint32_t *minmax) {
  double s = 0.0, c = 0.0;
  uint32_t lo = 0xFFFFFFFFu, hi = 0u;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float v = col[i];
    if (v == v) { s += (double)v; c += 1.0; const uint32_t k = f32_key(v); lo = min(lo, k); hi = max(hi, k); }
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o); c += __shfl_xor_sync(0xffffffffu, c, o);
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o)); hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out, s); atomicAdd(out + 1, c); atomicMin(minmax, lo); atomicMax(minmax + 1, hi); }
}

// max over a gp column (ignoring masked cells): sizes the lookup table
__global__ void colmax_u32_kernel(const uint32_t *__restrict__ col, size_t n, uint32_t *out) {
  uint32_t m = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const uint32_t v = col[i];
    if (v != GP_SENTINEL && v > m) m = v;
  }
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// ---------------------------------------------------------------------------
// Parameter build: everything that depends on (group, feature[, category]) but
// not on the row is evaluated once per sweep, in fp64, and laid out as the
// score kernel streams it: for k-tile t, feature d: chunk[rows_d][KT] floats.
// ---------------------------------------------------------------------------
__global__ void build_params_kernel(const FeatDev *__restrict__ feats, int nfeat, const double *__restrict__ hp,
                                    const double *__restrict__ ss, const int32_t *__restrict__ col2slot, int ncols,
                                    int KT, size_t region_rows, float *__restrict__ params, int tail_g) {
  // tail_g > 0: the columns of the last k-tile are replicated every tail_g floats (score kernel, ragged last tile)
  const int d = blockIdx.x, kt = blockIdx.y;
  const bool rep = tail_g > 0 && kt == (int)gridDim.y - 1;
  const FeatDev f = feats[d];
  if (f.rows == 0) return;
  float *chunk = params + ((size_t)kt * region_rows + f.rowoff) * KT;
  const double *fhp = hp + f.hp_off;
  const int total = (int)f.rows * KT;
  for (int i = blockIdx.z * blockDim.x + threadIdx.x; i < total; i += blockDim.x * gridDim.z) {  // z: slices of one chunk
    const int xr = i / KT, kl = i - xr * KT;
    const int col = kt * KT + (rep ? kl % tail_g : kl);
    float v = 0.f;
    if (col < ncols) {
      const double *gss = ss + f.ss_off + (size_t)col2slot[col] * f.ss_w;
      if (f.kind == KIND_TABLE && f.binform) {  // rows: t1 - t0 (difference taken in fp64), t0
        const double t0 = bb_score(fhp, gss, 0), t1 = bb_score(fhp, gss, 1);
        v = xr == 0 ? (float)(t1 - t0) : (float)t0;
      } else if (f.kind == KIND_TABLE) {
        if ((uint32_t)xr < f.ncat)
          v = (float)(f.family == FAM_BB ? bb_score(fhp, gss, xr) : f.family == FAM_BBNC ? bbnc_score(gss, xr)
                                                                                    : dd_score(fhp, f.asum, gss, (uint32_t)xr));
      } else if (f.kind == KIND_GP && f.family == FAM_BNB) {
        if ((uint32_t)xr < f.ncat) v = (float)bnb_score(bnb_post(fhp, gss), (double)xr);
      } else if (f.kind == KIND_GP) {
        const GpPost p = gp_post(fhp, gss);
        if ((uint32_t)xr < f.ncat) v = (float)gp_score(p, (double)xr);
        else if ((uint32_t)xr == f.ncat) v = 0.f;
        else if ((uint32_t)xr == f.ncat + 1) v = (float)p.a;
        else if ((uint32_t)xr == f.ncat + 2) v = (float)p.ca;
        else v = (float)p.l1pb;
      } else if (f.kind == KIND_NICH) {
        const NichPost p = nich_post(fhp, gss);
        // rows: mu' - c, s, c1 ln2 (the score kernel evaluates log2(1+z)), c0.  c is the centre of the score column
        // (msb_state_bind): for a column that sits far from 0 relative to its spread the fp32 table entry of mu'
        // would otherwise carry ulp(mu') of error into t = (x - mu') s
        v = xr == 0 ? (float)(p.mu - f.asum) : xr == 1 ? (float)p.s : xr == 2 ? (float)(p.c1 * 0.6931471805599453) : (float)p.c0;
      }
    }
    chunk[i] = v;
  }
}

// ---------------------------------------------------------------------------
// Direct scorer: closed forms straight from the suffstats in fp64, no tables.
// Used for single-entity score_value (entity_state.hpp:60-72) and as an
// independent on-device cross-check of the table path.  Scalar families only.
// ---------------------------------------------------------------------------
// OUT = float: the API's fp32 scores; OUT = double: the fp64 result itself (msb_state_score_rows_f64, held to 1e-12).
template <typename OUT>
__global__ void score_direct_kernel(const FeatDev *__restrict__ feats, int nfeat, const double *__restrict__ hp,
                                    const double *__restrict__ ss, const int32_t *__restrict__ col2slot, int ncols,
                                    const float *__restrict__ base, OUT *__restrict__ scores, size_t ld,
                                    size_t row_lo, size_t row_hi) {
  const size_t row = row_lo + blockIdx.x;
  if (row >= row_hi) return;
  for (int col = threadIdx.x; col < ncols; col += blockDim.x) {
    const int slot = col2slot[col];
    double s = 0.0;
    for (int d = 0; d < nfeat; d++) {
      const FeatDev f = feats[d];
      const double *fhp = hp + f.hp_off;
      const double *gss = ss + f.ss_off + (size_t)slot * f.ss_w;
      if (f.kind == KIND_TABLE) {
        uint32_t x;
        if (f.coltype == COL_U8) x = ((const uint8_t *)f.col)[row];
        else if (f.coltype == COL_U16) x = ((const uint16_t *)f.col)[row];
        else x = ((const uint32_t *)f.col)[row];
        if (x >= f.ncat) continue;
        s += f.family == FAM_BB ? bb_score(fhp, gss, (int)x) : f.family == FAM_BBNC ? bbnc_score(gss, (int)x) : dd_score(fhp, f.asum, gss, x);
      } else if (f.kind == KIND_GP) {
        const uint32_t x = ((const uint32_t *)f.col)[row];
        if (x == GP_SENTINEL) continue;
        s += f.family == FAM_BNB ? bnb_score(bnb_post(fhp, gss), (double)x) : gp_score(gp_post(fhp, gss), (double)x);
      } else if (f.kind == KIND_NICH) {
        const float x = ((const float *)f.col)[row];
        if (x != x) continue;
        s += nich_score(nich_post(fhp, gss), (double)x);
      }
    }
    scores[(row - row_lo) * ld + col] = (OUT)(s + (double)base[col]);
  }
}

// ---------------------------------------------------------------------------
// NIW: per-group preparation (posterior, Cholesky, inverse factor) in fp64.
//   hp = [mu[d], kappa, psi[d*d], nu]   ss = [count, sum_x[d], sum_xxT[d*d]]
// Outputs per column k: W[k] = L^-1 (row-major d x d, float), bias[k] = W mu',
// coef[k] = {c0, -(dof+d)/2, 1/dof}.  score = c0 + c1 log1p(|W x - bias|^2 / dof).
// ---------------------------------------------------------------------------
__global__ void niw_prepare_kernel(FeatDev f, const double *__restrict__ hp, const double *__restrict__ ss,
                                   const int32_t *__restrict__ col2slot, float *__restrict__ W,
                                   float *__restrict__ bias, float *__restrict__ coef) {
  extern __shared__ double sm[];
  const int d = (int)f.dim;
  double *A = sm;            // d*d
  double *mu = A + d * d;    // d
  double *Winv = mu + d;     // d*d
  __shared__ double s_logdiag;
  __shared__ int s_fail;
  const int k = blockIdx.x;
  const double *fhp = hp + f.hp_off;
  const double *gss = ss + f.ss_off + (size_t)col2slot[k] * f.ss_w;
  const double *mu0 = fhp, kappa0 = fhp[d], *psi0 = fhp + d + 1, nu0 = fhp[d + 1 + (size_t)d * d];
  const double n = gss[0];
  const double *sx = gss + 1, *sxx = gss + 1 + d;
  const double kn = kappa0 + n, nun = nu0 + n;
  const double dof = nun - (double)d + 1.0;
  const double scale = (kn + 1.0) / (kn * dof);
  if (threadIdx.x == 0) { s_fail = 0; s_logdiag = 0.0; }
  for (int i = threadIdx.x; i < d; i += blockDim.x) mu[i] = (kappa0 * mu0[i] + sx[i]) / kn;
  __syncthreads();
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) {
    const int i = e / d, j = e - i * d;
    A[e] = (psi0[e] + sxx[e] + kappa0 * mu0[i] * mu0[j] - kn * mu[i] * mu[j]) * scale;
  }
  __syncthreads();
  // right-looking Cholesky, lower triangle in place
  for (int j = 0; j < d; j++) {
    if (threadIdx.x == 0) {
      const double v = A[j * d + j];
      if (!(v > 0.0)) s_fail = 1;
      A[j * d + j] = sqrt(v > 0.0 ? v : 1.0);
    }
    __syncthreads();
    const double ljj = A[j * d + j];
    for (int i = j + 1 + threadIdx.x; i < d; i += blockDim.x) A[i * d + j] /= ljj;
    __syncthreads();
    // trailing update of the lower triangle: thread (ta, tb) of a 16 x (blockDim / 16) grid walks rows a and columns b <= a
    // (no integer division per element; the same subtraction per element as before, so the same bits)
    {
      const int tb = threadIdx.x & 15, ta = threadIdx.x >> 4, na = blockDim.x >> 4;
      for (int a = j + 1 + ta; a < d; a += na) {
        const double laj = A[a * d + j];
        for (int b = j + 1 + tb; b <= a; b += 16) A[a * d + b] -= laj * A[b * d + j];
      }
    }
    __syncthreads();
  }
  // W = L^-1: thread c solves L w = e_c by forward substitution, its column kept in registers / local order; the
  // reciprocal diagonal is NOT precomputed (t / L_ii as before: same bits)
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    for (int i = 0; i < c; i++) Winv[i * d + c] = 0.0;
    for (int i = c; i < d; i++) {
      double t = (i == c) ? 1.0 : 0.0;
      const double *Ai = A + i * d;
      for (int m = c; m < i; m++) t -= Ai[m] * Winv[m * d + c];
      Winv[i * d + c] = t / Ai[i];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ld = 0.0;
    for (int i = 0; i < d; i++) ld += log(A[i * d + i]);
    s_logdiag = ld;
  }
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) W[(size_t)k * d * d + e] = (float)Winv[e];
  // the scorers read the centred rows x - c (FeatDev::scol): bias = W (mu' - c)
  const float *cen = (const float *)f.slowmask;
  for (int i = threadIdx.x; i < d; i += blockDim.x) {
    double b = 0.0;
    for (int j = 0; j <= i; j++) b += Winv[i * d + j] * (mu[j] - (cen ? (double)cen[j] : 0.0));
    bias[(size_t)k * d + i] = (float)b;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const double c0 = lgamma(0.5 * (dof + d)) - lgamma(0.5 * dof) - 0.5 * d * log(dof * CUDART_PI) - s_logdiag;
    coef[(size_t)k * 4 + 0] = s_fail ? CUDART_NAN_F : (float)c0;
    coef[(size_t)k * 4 + 1] = (float)(-0.5 * (dof + d));
    coef[(size_t)k * 4 + 2] = (float)(1.0 / dof);
    coef[(size_t)k * 4 + 3] = 0.f;
  }
}

// ---------------------------------------------------------------------------
// group::score_data (models/base.hpp:28, forwarded at distributions.hpp:287-291): log marginal likelihood of the
// data a group holds, per (group column, feature), fp64 closed forms from the resident suffstats.
// out[col * nfeat + d].  K x D evaluations: not a hot kernel.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double lbeta_d(double a, double b) { return lgamma(a) + lgamma(b) - lgamma(a + b); }

__global__ void score_data_kernel(const FeatDev *__restrict__ feats, int nfeat, const double *__restrict__ hp,
                                  const double *__restrict__ ss, const int32_t *__restrict__ col2slot, int ncols,
                                  double *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ncols * nfeat) return;
  const int col = i / nfeat, d = i - col * nfeat;
  const FeatDev f = feats[d];
  if (f.kind == KIND_NIW) return;  // niw_score_data_kernel
  const double *h = hp + f.hp_off;
  const double *g = ss + f.ss_off + (size_t)col2slot[col] * f.ss_w;
  double r;
  if (f.family == FAM_DM) {  // dm.cpp:79-95; ss = [counts[dim], ratio]
    double asum = 0.0, csum = 0.0;
    r = g[f.dim];
    for (uint32_t c = 0; c < f.dim; c++) { asum += h[c]; csum += g[c]; r += lgamma(g[c] + h[c]) - lgamma(h[c]); }
    r += lgamma(asum) - lgamma(asum + csum);
  } else if (f.family == FAM_BB) {
    r = lbeta_d(h[0] + g[0], h[1] + g[1]) - lbeta_d(h[0], h[1]);
  } else if (f.family == FAM_BBNC) {  // bbnc.cpp:61-73: Beta prior density of p + Bernoulli likelihood of the counts
    const double p = g[0];
    r = (p < 0.0 || p > 1.0) ? -CUDART_INF
                             : (h[0] - 1.0) * log(p) + (h[1] - 1.0) * log1p(-p) - lbeta_d(h[0], h[1]) + g[1] * log(p) + g[2] * log1p(-p);
  } else if (f.family == FAM_DD) {
    r = lgamma(f.asum) - lgamma(f.asum + g[0]);
    for (uint32_t c = 0; c < f.dim; c++) r += lgamma(h[c] + g[1 + c]) - lgamma(h[c]);
  } else if (f.family == FAM_BNB) {
    // (count, sum) do not determine sum_i [lgamma(r + x_i) - lgamma(r) - lgamma(x_i + 1)]: like the family's own
    // two-field group this returns the part that depends on the partition and on (alpha, beta)
    const double a = h[0] + h[2] * g[0], b = h[1] + g[1];
    r = lbeta_d(a, b) - lbeta_d(h[0], h[1]);
  } else if (f.kind == KIND_GP) {  // prior Gamma(alpha, rate inv_beta); ss = count, sum, sum log x!
    const double a = h[0] + g[1], b = h[1] + g[0];
    r = lgamma(a) - lgamma(h[0]) + h[0] * log(h[1]) - a * log(b) - g[2];
  } else {  // nich; device ss = (count, sum x, sum x^2)
    const double n = g[0];
    const double mean = n > 0.0 ? g[1] / n : 0.0;
    double ctv = n > 0.0 ? g[2] - g[1] * mean : 0.0;
    if (ctv < 0.0) ctv = 0.0;
    const double mu1 = h[0] - mean;
    const double kappa = h[1] + n, nu = h[3] + n;
    const double sigmasq = (h[3] * h[2] + ctv + (n * h[1] * mu1 * mu1) / kappa) / nu;
    r = lgamma(0.5 * nu) - lgamma(0.5 * h[3]) + 0.5 * log(h[1] / kappa) + 0.5 * h[3] * log(h[3] * h[2]) -
        0.5 * nu * log(nu * sigmasq) - 0.5 * n * log(CUDART_PI);
  }
  out[i] = r;
}

// In-place lower Cholesky of the d x d matrix A in shared memory by the whole block (right-looking, as in
// niw_prepare_kernel); returns log |A| = 2 sum log L_ii, NaN if A is not positive definite.
__device__ double block_chol_logdet(double *A, int d, int *s_fail, double *s_acc) {
  if (threadIdx.x == 0) { *s_fail = 0; *s_acc = 0.0; }
  __syncthreads();
  for (int j = 0; j < d; j++) {
    if (threadIdx.x == 0) {
      const double v = A[j * d + j];
      if (!(v > 0.0)) *s_fail = 1;
      A[j * d + j] = sqrt(v > 0.0 ? v : 1.0);
      *s_acc += 2.0 * log(A[j * d + j]);
    }
    __syncthreads();
    const double ljj = A[j * d + j];
    for (int i = j + 1 + threadIdx.x; i < d; i += blockDim.x) A[i * d + j] /= ljj;
    __syncthreads();
    const int rem = d - j - 1;
    for (int e = threadIdx.x; e < rem * rem; e += blockDim.x) {
      const int a = j + 1 + e / rem, b = j + 1 + e % rem;
      if (b <= a) A[a * d + b] -= A[a * d + j] * A[b * d + j];
    }
    __syncthreads();
  }
  return *s_fail ? CUDART_NAN : *s_acc;
}

// NIW marginal likelihood, one block per group column:
//   -n d/2 log pi + lgamma_d(nu'/2) - lgamma_d(nu/2) + nu/2 log|psi| - nu'/2 log|psi'| + d/2 log(kappa/kappa')
__global__ void niw_score_data_kernel(FeatDev f, int feat_index, int nfeat, const double *__restrict__ hp,
                                      const double *__restrict__ ss, const int32_t *__restrict__ col2slot,
                                      double *__restrict__ out) {
  extern __shared__ double sm[];
  const int d = (int)f.dim;
  double *A = sm;          // d*d
  double *mu = A + d * d;  // d
  __shared__ int s_fail;
  __shared__ double s_acc;
  const int k = blockIdx.x;
  const double *fhp = hp + f.hp_off;
  const double *gss = ss + f.ss_off + (size_t)col2slot[k] * f.ss_w;
  const double *mu0 = fhp, kappa0 = fhp[d], *psi0 = fhp + d + 1, nu0 = fhp[d + 1 + (size_t)d * d];
  const double n = gss[0];
  const double *sx = gss + 1, *sxx = gss + 1 + d;
  const double kn = kappa0 + n, nun = nu0 + n;
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) A[e] = psi0[e];
  __syncthreads();
  const double ld0 = block_chol_logdet(A, d, &s_fail, &s_acc);
  __syncthreads();
  for (int i = threadIdx.x; i < d; i += blockDim.x) mu[i] = (kappa0 * mu0[i] + sx[i]) / kn;
  __syncthreads();
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) {
    const int i = e / d, j = e - i * d;
    A[e] = psi0[e] + sxx[e] + kappa0 * mu0[i] * mu0[j] - kn * mu[i] * mu[j];
  }
  __syncthreads();
  const double ldn = block_chol_logdet(A, d, &s_fail, &s_acc);
  if (threadIdx.x == 0) {
    double lg = 0.0;  // lgamma_d(nu'/2) - lgamma_d(nu/2): the pi^(d(d-1)/4) factors cancel
    for (int j = 0; j < d; j++) lg += lgamma(0.5 * (nun - j)) - lgamma(0.5 * (nu0 - j));
    out[(size_t)k * nfeat + feat_index] = -0.5 * n * d * log(CUDART_PI) + lg + 0.5 * nu0 * ld0 - 0.5 * nun * ldn +
                                          0.5 * d * log(kappa0 / kn);
  }
}

// group_manager::score_assignment (group_manager.hpp:250-272) in closed form from the resident counts: the CRP
// probability of a partition depends only on the group sizes and on which group holds entity 0:
//   sum_g [log alpha (unless g holds entity 0) + lgamma(n_g)] - (lgamma(n + alpha) - lgamma(1 + alpha)).
// out[0] = the score, out[1] = number of assigned entities (the caller checks it equals n).  One block.
__global__ void score_assignment_kernel(const double *__restrict__ counts, const int32_t *__restrict__ col2slot,
                                        int ncols, const int32_t *__restrict__ assign, double alpha,
                                        double *__restrict__ out) {
  __shared__ double s_sum, s_n;
  if (threadIdx.x == 0) { s_sum = 0.0; s_n = 0.0; }
  __syncthreads();
  const int first = assign[0];
  double s = 0.0, n = 0.0;
  for (int c = threadIdx.x; c < ncols; c += blockDim.x) {
    const int slot = col2slot[c];
    const double cnt = counts[slot];
    if (cnt > 0.0) {
      s += (slot == first ? 0.0 : log(alpha)) + lgamma(cnt);
      n += cnt;
    }
  }
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); n += __shfl_xor_sync(0xffffffffu, n, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(&s_sum, s); atomicAdd(&s_n, n); }
  __syncthreads();
  if (threadIdx.x == 0) {
    out[0] = s_sum - (lgamma(s_n + alpha) - lgamma(1.0 + alpha));
    out[1] = s_n;
  }
}

// ---------------------------------------------------------------------------
// dm (Dirichlet-multinomial over count vectors, src/models/dm.cpp:38-76).  One block per group column: the block
// holds e_i = alpha_i + counts_i in shared memory, each thread scores rows:
//   sum_i [lgamma(e_i + x_i) - lgamma(e_i) - lgamma(x_i + 1)] + lgamma(X + 1) + lgamma(E) - lgamma(E + X)
// scores[(row - row_lo) * ld + k] += that (OUT = float: the production path; OUT = double: the fp64 path).
// ---------------------------------------------------------------------------
template <typename OUT>
__global__ void dm_score_kernel(FeatDev f, const double *__restrict__ hp, const double *__restrict__ ss,
                                const int32_t *__restrict__ col2slot, OUT *__restrict__ scores, size_t ld,
                                size_t row_lo, size_t row_hi) {
  extern __shared__ double sm[];
  const int C = (int)f.dim;
  double *e = sm;  // C
  __shared__ double s_E;
  const int k = blockIdx.y;
  const double *h = hp + f.hp_off;
  const double *g = ss + f.ss_off + (size_t)col2slot[k] * f.ss_w;
  for (int i = threadIdx.x; i < C; i += blockDim.x) e[i] = h[i] + g[i];
  __syncthreads();
  if (threadIdx.x == 0) { double E = 0.0; for (int i = 0; i < C; i++) E += e[i]; s_E = E; }
  __syncthreads();
  const double E = s_E, lgE = lgamma(E);
  const size_t row = row_lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= row_hi) return;
  const uint32_t *x = (const uint32_t *)f.col + row * (size_t)C;
  if (x[0] == GP_SENTINEL) return;  // masked
  double s = 0.0, X = 0.0;
  for (int i = 0; i < C; i++) {
    const uint32_t xi = x[i];
    if (xi) { s += lgamma_rise(e[i], xi) - lgamma((double)xi + 1.0); X += (double)xi; }
  }
  s += lgamma(X + 1.0) + lgE - lgamma(E + X);
  scores[(row - row_lo) * ld + k] += (OUT)s;
}

// The batched form: a block owns a tile of 32 group columns (e_i transposed into shared memory, lane = group) and
// DM_TILE_ROWS rows (one warp per row, the row's counts are warp-uniform loads).  Per (row, group) the predictive is
//   log [ prod_i (e_i)_(x_i) / (E)_(X) ] + log X! - sum_i log x_i!      ((a)_(n) = a (a + 1) ... (a + n - 1))
// with the rising factorials multiplied out in fp64 (no lgamma(e + x) - lgamma(e) cancellation, one log per
// (row, group) instead of one per category) whenever the counts are small; large counts take the lgamma form.
constexpr int DM_TILE_ROWS = 64;
__constant__ double c_lfact[21] = {0.0, 0.0, 0.6931471805599453, 1.791759469228055, 3.1780538303479458, 4.787491742782046,
                                   6.579251212010101, 8.525161361065415, 10.604602902745251, 12.801827480081469,
                                   15.104412573075516, 17.502307845873887, 19.987214495661885, 22.552163853123425,
                                   25.19122118273868, 27.89927138384089, 30.671860106080672, 33.50507345013689,
                                   36.39544520803305, 39.339884187199495, 42.335616460753485};
__device__ __forceinline__ double lfact(uint32_t n) { return n <= 20u ? c_lfact[n] : lgamma((double)n + 1.0); }

template <typename OUT>
__global__ void __launch_bounds__(256) dm_score_tile_kernel(FeatDev f, const double *__restrict__ hp, const double *__restrict__ ss,
                                                            const int32_t *__restrict__ col2slot, int K, OUT *__restrict__ scores,
                                                            size_t ld, size_t row_lo, size_t row_hi) {
  extern __shared__ double sm[];
  const int C = (int)f.dim;
  double *eT = sm;            // [C][32]
  double *Es = sm + C * 32;   // [32]: E = sum_i e_i
  double *lgE = Es + 32;      // [32]
  const int k0 = blockIdx.y * 32;
  const double *h = hp + f.hp_off;
  for (int idx = threadIdx.x; idx < C * 32; idx += blockDim.x) {
    const int kk = idx / C, i = idx - kk * C;
    const int k = k0 + kk;
    eT[i * 32 + kk] = k < K ? h[i] + ss[f.ss_off + (size_t)col2slot[k] * f.ss_w + i] : 1.0;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    double E = 0.0;
    for (int i = 0; i < C; i++) E += eT[i * 32 + threadIdx.x];
    Es[threadIdx.x] = E;
    lgE[threadIdx.x] = lgamma(E);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = k0 + lane;
  const size_t tile_lo = row_lo + (size_t)blockIdx.x * DM_TILE_ROWS;
  const size_t tile_hi = tile_lo + DM_TILE_ROWS < row_hi ? tile_lo + DM_TILE_ROWS : row_hi;
  const double E = Es[lane];
  for (size_t row = tile_lo + warp; row < tile_hi; row += 8) {
    const uint32_t *x = (const uint32_t *)f.col + row * (size_t)C;
    if (x[0] == GP_SENTINEL) continue;  // masked (warp-uniform)
    double s = 0.0, p = 1.0, rowc = 0.0, X = 0.0;
    for (int i = 0; i < C; i++) {
      const uint32_t xi = x[i];
      if (!xi) continue;
      rowc -= lfact(xi);
      X += (double)xi;
      const double e = eT[i * 32 + lane];
      if (xi <= 12u) {
        for (uint32_t j = 0; j < xi; j++) p *= e + (double)j;
        if (p > 1e100 || p < 1e-100) { s += log(p); p = 1.0; }
      } else {
        s += lgamma(e + (double)xi) - lgamma(e);
      }
    }
    if (X <= 16.0) {
      double q = 1.0;
      const int n = (int)X;
      for (int j = 0; j < n; j++) q *= E + (double)j;
      s += log(p) - log(q);
    } else {
      s += log(p) + lgE[lane] - lgamma(E + X);
    }
    rowc += X <= 20.0 ? c_lfact[(int)X] : lgamma(X + 1.0);
    if (k < K) scores[(row - row_lo) * ld + k] += (OUT)(s + rowc);
  }
}

// dm update: one warp per moved row, lanes over the categories; counts += / -= x, ratio as dm.cpp:9-36
__global__ void update_dm_kernel(FeatDev f, const int32_t *__restrict__ old_slot, const int32_t *__restrict__ new_slot,
                                 size_t row_lo, size_t row_hi, double *__restrict__ delta) {
  const size_t row = row_lo + (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= row_hi) return;
  const int a = old_slot ? old_slot[row] : -1;
  const int b = new_slot ? new_slot[row - row_lo] : -1;
  if (a == b) return;
  const int C = (int)f.dim;
  const uint32_t *x = (const uint32_t *)f.col + row * (size_t)C;
  if (x[0] == GP_SENTINEL) return;
  double *blk = delta + f.ss_off;
  double part = 0.0, X = 0.0;  // sum lgamma(x_i + 1), sum x_i over this lane's categories
  for (int i = lane; i < C; i += 32) {
    const double xi = (double)x[i];
    if (xi != 0.0) {
      if (a >= 0) atomic_add_f64(blk + (size_t)a * f.ss_w + i, -xi);
      if (b >= 0) atomic_add_f64(blk + (size_t)b * f.ss_w + i, xi);
      part += lgamma(xi + 1.0);
      X += xi;
    }
  }
  for (int o = 16; o > 0; o >>= 1) { part += __shfl_xor_sync(0xffffffffu, part, o); X += __shfl_xor_sync(0xffffffffu, X, o); }
  if (lane == 0) {
    const double r = lgamma(X + 1.0) - part;  // add_value: ratio += lgamma(X + 1) - sum lgamma(x_i + 1)
    if (a >= 0) atomic_add_f64(blk + (size_t)a * f.ss_w + C, -r);
    if (b >= 0) atomic_add_f64(blk + (size_t)b * f.ss_w + C, r);
  }
}

// fp64 NIW scorer (verification path, any dim): one block per group column; the block factors the scale matrix
// (as niw_prepare_kernel does), then each thread scores rows by forward substitution in fp64.
// scores[(row - row_lo) * ld + k] += c0 - (dof + d)/2 log1p(|L^-1 (x - mu')|^2 / dof)
__global__ void niw_score_f64_kernel(FeatDev f, const double *__restrict__ hp, const double *__restrict__ ss,
                                     const int32_t *__restrict__ col2slot, double *__restrict__ scores, size_t ld,
                                     size_t row_lo, size_t row_hi) {
  extern __shared__ double sm[];
  const int d = (int)f.dim;
  double *A = sm;          // d*d: scale matrix, then its lower Cholesky factor
  double *mu = A + d * d;  // d
  __shared__ int s_fail;
  __shared__ double s_acc;
  const int k = blockIdx.x;
  const double *fhp = hp + f.hp_off;
  const double *gss = ss + f.ss_off + (size_t)col2slot[k] * f.ss_w;
  const double *mu0 = fhp, kappa0 = fhp[d], *psi0 = fhp + d + 1, nu0 = fhp[d + 1 + (size_t)d * d];
  const double n = gss[0];
  const double *sx = gss + 1, *sxx = gss + 1 + d;
  const double kn = kappa0 + n, nun = nu0 + n;
  const double dof = nun - (double)d + 1.0;
  const double scale = (kn + 1.0) / (kn * dof);
  for (int i = threadIdx.x; i < d; i += blockDim.x) mu[i] = (kappa0 * mu0[i] + sx[i]) / kn;
  __syncthreads();
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) {
    const int i = e / d, j = e - i * d;
    A[e] = (psi0[e] + sxx[e] + kappa0 * mu0[i] * mu0[j] - kn * mu[i] * mu[j]) * scale;
  }
  __syncthreads();
  const double logdet = block_chol_logdet(A, d, &s_fail, &s_acc);  // = 2 sum log L_ii
  const double c0 = lgamma(0.5 * (dof + d)) - lgamma(0.5 * dof) - 0.5 * d * log(dof * CUDART_PI) - 0.5 * logdet;
  for (size_t row = row_lo + threadIdx.x; row < row_hi; row += blockDim.x) {
    const float *x = (const float *)f.col + row * (size_t)d;
    if (x[0] != x[0]) continue;  // masked
    double q = 0.0;
    double y[96];
    for (int i = 0; i < d; i++) {
      double t = (double)x[i] - mu[i];
      for (int m = 0; m < i; m++) t -= A[i * d + m] * y[m];
      y[i] = t / A[i * d + i];
      q += y[i] * y[i];
    }
    scores[(row - row_lo) * ld + k] += c0 - 0.5 * (dof + d) * log1p(q / dof);
  }
}

// CUDA-core NIW scorer (any dim): thread per row, W_k staged in shared memory.
// scores[row][k] += c0 + c1 log1p(q / dof).  The tcgen05 path replaces this
// for dim == 64 (msb_niw_tc.cuh).
__global__ void niw_score_simt_kernel(const float *__restrict__ X, int d, const float *__restrict__ W,
                                      const float *__restrict__ bias, const float *__restrict__ coef,
                                      float *__restrict__ scores, size_t ld, size_t row_lo, size_t row_hi) {
  extern __shared__ float smf[];
  float *Wk = smf;          // d*d
  float *bk = Wk + d * d;   // d
  const int k = blockIdx.y;
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) Wk[e] = W[(size_t)k * d * d + e];
  for (int e = threadIdx.x; e < d; e += blockDim.x) bk[e] = bias[(size_t)k * d + e];
  __syncthreads();
  const size_t row = row_lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= row_hi) return;
  const float *x = X + row * (size_t)d;
  if (x[0] != x[0]) return;  // masked
  float q = 0.f;
  for (int i = 0; i < d; i++) {
    float y = -bk[i];
    for (int j = 0; j <= i; j++) y = fmaf(Wk[i * d + j], x[j], y);
    q = fmaf(y, y, q);
  }
  const float c0 = coef[(size_t)k * 4 + 0], c1 = coef[(size_t)k * 4 + 1], idof = coef[(size_t)k * 4 + 2];
  scores[(row - row_lo) * ld + k] += c0 + c1 * log1pf(q * idof);
}

// ---------------------------------------------------------------------------
// Sampler: util.hpp:125-156 exactly -- max, exp, double accumulation in group
// order, float division, sequential dart subtraction with last-index fallback.
// The order of the floating-point operations is part of the contract (the
// checker must reproduce the draw bit for bit), so one thread walks one row.
// ---------------------------------------------------------------------------
//
// The inverse-CDF walk `dart -= p / acc; if (dart <= 0) return k` is the only serial part.  dart_walk does it
// eight elements at a time: the eight quotients are independent (computed first), then eight FSUB/compare
// steps; the warp leaves once every lane has crossed zero.  The quotient RN(p / acc) is computed by Markstein's
// sequence with the correctly rounded reciprocal y = RN(1 / acc):
//     q0 = RN(p y),  r = RN(p - acc q0) (exact, FMA),  q = RN(q0 + r y)
// which equals the IEEE division whenever no intermediate underflows: p >= 2^-100 or p == 0, acc in [1, 2^24]
// (checked against exact rational arithmetic in tests/test_division_sequence.py and against __fdiv_rn on the
// device by msb_selftest_division).  A smaller non-zero p gives q < 2^-100, which cannot change a dart >= 2^-60;
// a batch in which a lane meets such a p with a smaller dart (or an acc outside the range) is redone with
// __fdiv_rn.  __fdiv_rn on every element would take its out-of-line slow path for every zero / subnormal p,
// i.e. on most elements of a well-separated mixture.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float div_markstein(float p, float acc, float y) {
  const float q0 = __fmul_rn(p, y);
  const float r = __fmaf_rn(-acc, q0, p);
  return __fmaf_rn(r, y, q0);
}

// the same sequence two quotients at a time (FMUL2 / FFMA2): the same roundings as div_markstein (a multiply feeding
// an FFMA2 has nothing ptxas could contract it with)
__device__ __forceinline__ float2 div_markstein2(float2 p, float acc, float y) {
  const float2 y2 = make_float2(y, y);
  const float2 q0 = __fmul2_rn(p, y2);
  const float2 r = __ffma2_rn(make_float2(-acc, -acc), q0, p);
  return __ffma2_rn(r, y2, q0);
}

// Sparsity: exp(s - max) underflows to exactly 0 below -104, which in a mixture is the case for most groups of
// most rows.  A batch of eight groups whose p is exactly 0 in every lane of the warp leaves every live dart
// unchanged (dart - 0), so it is skipped as a whole (dead8(k0), warp-uniform); the same test lets the exp pass
// skip the polynomial (exp_is_zero).  Results are bit-identical, only the work drops.
__device__ __forceinline__ bool exp_is_zero(float x) { return x < -104.0f; }  // false for NaN, like msb_expf

// The walk's exact skip (DESIGN.md section 4.3): a dart d >= 2^-60 stays bit for bit, and so makes no pick, over a batch
// whose largest p has the biased exponent e (every p < 2^(e - 126)) when acc is in [1, 2^24] and e <= Ea + Ed - 154
// (Ea, Ed: the biased exponents of acc and d): then every RN(p / acc) is below half the spacing of the floats just
// below d.  e = 255 (a NaN p) never passes.
__device__ __forceinline__ bool dart_keeps(uint32_t e, float acc, float d) {
  return acc >= 1.0f && acc <= 16777216.0f && d >= 0x1p-60f &&
         (int)e <= (__float_as_int(acc) >> 23) - 154 + (__float_as_int(d) >> 23);
}

// all 32 lanes of the warp must call this (lanes without a row pass found = true).
// skip8(k0, found, dart): this lane's dart and pick provably stay as they are over the batch k0 .. k0 + 7; the batch
// is skipped when that holds in every lane.  PADDED: p_of(k) is +0 for K <= k < K rounded up to 8.
template <bool PADDED = false, typename F, typename G>
__device__ __forceinline__ void dart_walk(int K, float acc, float dart, bool found, int &pick, F p_of, G skip8) {
  const float y = __frcp_rn(acc);
  const bool odd = !(acc >= 1.0f && acc <= 16777216.0f);
  pick = K - 1;
  for (int k0 = 0; k0 < K; k0 += 8) {
    if (__all_sync(0xffffffffu, skip8(k0, found, dart))) continue;
    float p[8], q[8];
#pragma unroll
    for (int j = 0; j < 8; j++) p[j] = PADDED || k0 + j < K ? p_of(k0 + j) : 0.f;
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      const float2 qq = div_markstein2(make_float2(p[j], p[j + 1]), acc, y);
      q[j] = qq.x; q[j + 1] = qq.y;
    }
    const float dart0 = dart;
    const int pick0 = pick;
    const bool found0 = found;
    bool suspect = odd && !found;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      suspect |= !found && dart < 0x1p-60f && p[j] < 0x1p-100f && p[j] > 0.f;
      dart = __fsub_rn(dart, q[j]);
      // a padding element (p = +0) cannot make the pick: a dart not found before it is > 0 or NaN and stays so
      if (!found && dart <= 0.f && (PADDED || k0 + j < K)) { pick = k0 + j; found = true; }
    }
    if (__any_sync(0xffffffffu, suspect)) {  // rare: redo the batch with the IEEE division
      dart = dart0; pick = pick0; found = found0;
#pragma unroll 1
      for (int j = 0; j < 8; j++) {
        if (k0 + j >= K) break;
        dart = __fsub_rn(dart, __fdiv_rn(p_of(k0 + j), acc));
        if (!found && dart <= 0.f) { pick = k0 + j; found = true; }
      }
    }
    if (__all_sync(0xffffffffu, found)) break;
  }
}

__global__ void sample_kernel(const float *__restrict__ scores, size_t ld, int K, size_t nrows,
                              const float *__restrict__ uniforms, uint64_t seed, uint64_t sweep, uint64_t row_id0,
                              const int32_t *__restrict__ col2slot, int32_t *__restrict__ out_col,
                              int32_t *__restrict__ out_slot) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < nrows;
  const float *s = scores + (valid ? i : 0) * ld;
  float m = s[0];
  for (int k = 1; k < K; k++) m = fmaxf(m, s[k]);
  auto dead8 = [&](int k0) {
    bool live = false;
#pragma unroll
    for (int j = 0; j < 8; j++) live |= k0 + j < K && !exp_is_zero(__fsub_rn(s[k0 + j], m));
    return !__any_sync(0xffffffffu, live);
  };
  double acc_d = 0.0;
  for (int k0 = 0; k0 < K; k0 += 8) {
    if (dead8(k0)) continue;  // acc + 0 = acc
#pragma unroll
    for (int j = 0; j < 8; j++)
      if (k0 + j < K) acc_d = __dadd_rn(acc_d, (double)msb_expf(__fsub_rn(s[k0 + j], m)));
  }
  const float acc = __double2float_rn(acc_d);
  float dart = 0.f;
  if (valid) dart = uniforms ? uniforms[i] : philox_u01(seed, row_id0 + i, sweep);
  int pick;
  // every p of a dead batch is +0 in every lane: q = +0 and dart - 0 = dart, unless a lane sits exactly on dart <= 0
  dart_walk(K, acc, dart, !valid, pick, [&](int k) { return msb_expf(__fsub_rn(s[k], m)); },
            [&](int k0, bool f, float d) { return dead8(k0) && (f || d > 0.f); });
  if (!valid) return;
  if (out_col) out_col[i] = pick;
  if (out_slot) out_slot[i] = col2slot ? col2slot[pick] : pick;
}

// The same walk over the blocked layout the sweep's score kernel writes (msb_score.cuh): thread =
// row, element k of the row at s[k * 32]; every load is a fully coalesced 128-byte warp access.
__global__ void sample_blocked_kernel(const float *__restrict__ scores, size_t ld, size_t skip, int K, size_t nrows,
                                      const float *__restrict__ uniforms, uint64_t seed, uint64_t sweep,
                                      uint64_t row_id0, const int32_t *__restrict__ col2slot,
                                      int32_t *__restrict__ out_col, int32_t *__restrict__ out_slot,
                                      const int *__restrict__ rowmax) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < nrows;
  const size_t loc = (valid ? i : 0) + skip;  // position in the buffer, whose origin is a multiple of 128 rows
  const float *s = scores + (loc / 32) * ld * 32 + (loc % 32);
  float m;
  if (rowmax) {
    // the score kernel's epilogue left the row's maximum (score_bundle_kernel): the same floats, the same maximum, one
    // pass over the score matrix less
    int ord = rowmax[loc];
    m = ord == (int)0x80808080 ? s[0] : __int_as_float(ord ^ ((ord >> 31) & 0x7fffffff));   // (never written: a row outside the scored range)
  } else {
    float m0 = s[0], m1 = m0, m2 = m0, m3 = m0;
    int k = 1;
    for (; k + 3 < K; k += 4) {
      m0 = fmaxf(m0, s[(size_t)k * 32]); m1 = fmaxf(m1, s[(size_t)(k + 1) * 32]);
      m2 = fmaxf(m2, s[(size_t)(k + 2) * 32]); m3 = fmaxf(m3, s[(size_t)(k + 3) * 32]);
    }
    for (; k < K; k++) m0 = fmaxf(m0, s[(size_t)k * 32]);
    m = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
  }
  auto dead8 = [&](int k0) {
    bool live = false;
#pragma unroll
    for (int j = 0; j < 8; j++) live |= k0 + j < K && !exp_is_zero(__fsub_rn(s[(size_t)(k0 + j) * 32], m));
    return !__any_sync(0xffffffffu, live);
  };
  // Which batches of eight groups are alive is found out in the sum pass and REMEMBERED (one bit per batch, warp-
  // uniform, up to 256 batches = K <= 2048 in four registers), so that the walk neither re-reads the dead batches to
  // test them again nor touches their memory at all: in a separated mixture (C3: 99.8 % of the elements dead) the third
  // pass over the score matrix -- a third of this kernel's DRAM traffic, which at K > 384 no cache holds -- shrinks to
  // the live batches.  Larger K falls back to testing again.
  const bool remember = K <= 2048;
  uint64_t l0 = 0, l1 = 0, l2 = 0, l3 = 0;
  double acc_d = 0.0;
  for (int k0 = 0; k0 < K; k0 += 8) {
    if (dead8(k0)) continue;  // acc + 0 = acc
    const int b = k0 >> 3;
    const uint64_t bit = 1ull << (b & 63);
    if (b < 64) l0 |= bit; else if (b < 128) l1 |= bit; else if (b < 192) l2 |= bit; else l3 |= bit;
#pragma unroll
    for (int j = 0; j < 8; j++)
      if (k0 + j < K) acc_d = __dadd_rn(acc_d, (double)msb_expf(__fsub_rn(s[(size_t)(k0 + j) * 32], m)));
  }
  const float acc = __double2float_rn(acc_d);
  float dart = 0.f;
  if (valid) dart = uniforms ? uniforms[i] : philox_u01(seed, row_id0 + i, sweep);
  int pick;
  auto dead8_known = [&](int k0) {
    if (!remember) return dead8(k0);
    const int b = k0 >> 3;
    const uint64_t w = b < 64 ? l0 : (b < 128 ? l1 : (b < 192 ? l2 : l3));
    return !((w >> (b & 63)) & 1ull);
  };
  dart_walk(K, acc, dart, !valid, pick, [&](int kk) { return msb_expf(__fsub_rn(s[(size_t)kk * 32], m)); },
            [&](int k0, bool f, float d) { return dead8_known(k0) && (f || d > 0.f); });
  if (!valid) return;
  if (out_col) out_col[i] = pick;
  if (out_slot) out_slot[i] = col2slot ? col2slot[pick] : pick;
}

// y[i] = msb_expf(x[i]): device self-test against the checker's separately written copy
__global__ void selftest_expf_kernel(const float *__restrict__ x, size_t n, float *__restrict__ y) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = msb_expf(x[i]);
}

// msb_expf2_dense against msb_expf on every float of [-86, 0]: thread t takes the pair -f(2t), -f(2t + 1), where f(b)
// is the float with the bits b (b = 0 is -0); the last thread takes -86 and +0.  Counts the differing results.
constexpr uint32_t EXPF2_LAST_BITS = 0x42AC0000u;  // 86.0f (even)
__global__ void selftest_expf2_kernel(unsigned long long *mismatches) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > EXPF2_LAST_BITS / 2) return;
  float2 x = make_float2(-__uint_as_float(2 * t), -__uint_as_float(2 * t + 1));
  if (t == EXPF2_LAST_BITS / 2) x = make_float2(-86.0f, 0.0f);
  const float2 y = msb_expf2_dense(x);
  const unsigned bad = (__float_as_uint(y.x) != __float_as_uint(msb_expf(x.x))) +
                       (__float_as_uint(y.y) != __float_as_uint(msb_expf(x.y)));
  if (bad) atomicAdd(mismatches, (unsigned long long)bad);
}

// q[i] = (a[i] / b[i] by Markstein's sequence) != __fdiv_rn(a[i], b[i]) counted: device self-test of dart_walk's
// division, scalar and packed, on pseudo-random operands p in [2^-100, 1], acc in [1, 2^24) (plus exact zeros)
__global__ void selftest_division_kernel(uint64_t seed, size_t n, unsigned long long *mismatches) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t r[4];
  philox4x32_10(seed, i, 0x5e1f7e57ull, r);
  // p: random mantissa, exponent in [-100, 0]; every 64th operand is an exact zero
  const uint32_t pe = 127 - (r[2] % 101);
  float p = __uint_as_float((pe << 23) | (r[0] & 0x7fffffu));
  if (p > 1.0f) p = 1.0f;
  if ((r[3] & 63u) == 0) p = 0.f;
  const uint32_t ae = 127 + ((r[2] >> 8) % 24);
  const float acc = __uint_as_float((ae << 23) | (r[1] & 0x7fffffu));
  // a second dividend for the packed form the walk uses: another mantissa and exponent from the same block
  float p2 = __uint_as_float(((127 - ((r[3] >> 8) % 101)) << 23) | (r[3] >> 9));
  if (p2 > 1.0f) p2 = 1.0f;
  if ((r[3] & 0xFC0u) == 0) p2 = 0.f;
  const float y = __frcp_rn(acc);
  const float got = div_markstein(p, acc, y);
  const float2 got2 = div_markstein2(make_float2(p, p2), acc, y);
  const float want = __fdiv_rn(p, acc), want2 = __fdiv_rn(p2, acc);
  const unsigned bad = (__float_as_uint(got) != __float_as_uint(want)) + (__float_as_uint(got2.x) != __float_as_uint(want)) +
                       (__float_as_uint(got2.y) != __float_as_uint(want2));
  if (bad) atomicAdd(mismatches, (unsigned long long)bad);
}

// out[i] = dart_keeps(e[i], acc[i], d[i]): the walk's skip test on given operands, for the exact check on the host
__global__ void selftest_skip_rule_kernel(const uint8_t *__restrict__ e, const float *__restrict__ acc,
                                          const float *__restrict__ d, size_t n, uint8_t *__restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = dart_keeps(e[i], acc[i], d[i]) ? 1 : 0;
}

// blocked -> row-major copy of a score matrix (diagnostics / tests)
__global__ void unblock_kernel(const float *__restrict__ blocked, size_t ld, size_t skip, size_t nrows, int K,
                               float *__restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nrows * (size_t)K) return;
  const size_t row = i / K + skip, col = i % K;
  out[i] = blocked[((row / 32) * ld + col) * 32 + (row % 32)];
}

__global__ void philox_fill_kernel(uint64_t seed, uint64_t sweep, uint64_t row0, size_t n, float *out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = philox_u01(seed, row0 + i, sweep);
}

// ---------------------------------------------------------------------------
// Suffstat update: remove_value(old group) / add_value(new group) for every
// (row, feature) cell whose row moved (base.hpp:25-26).  All device suffstats
// are additive fp64 (integers exact), so the deltas can be summed across GPUs.
// ---------------------------------------------------------------------------

constexpr int UPDATE_SLAB = 16;
__global__ void update_kernel(const FeatDev *__restrict__ feats, int nfeat, const int32_t *__restrict__ old_slot,
                              const int32_t *__restrict__ new_slot, size_t row_lo, size_t row_hi,
                              double *__restrict__ delta) {
  // thread = row; blockIdx.y = a slab of UPDATE_SLAB features: the two assignment loads are shared by the slab,
  // a row that did not move costs nothing more, and for a fixed feature the column loads of a warp are coalesced
  const size_t row = row_lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= row_hi) return;
  const int a = old_slot ? old_slot[row] : -1;
  const int b = new_slot ? new_slot[row - row_lo] : -1;
  if (a == b) return;
  const int d_hi = min(nfeat, (int)(blockIdx.y + 1) * UPDATE_SLAB);
  for (int d = blockIdx.y * UPDATE_SLAB; d < d_hi; d++) {
    const FeatDev &f = feats[d];
    double *blk = delta + f.ss_off;
    if (f.kind == KIND_TABLE) {
      uint32_t x;
      if (f.coltype == COL_U8) x = ((const uint8_t *)f.col)[row];
      else if (f.coltype == COL_U16) x = ((const uint16_t *)f.col)[row];
      else x = ((const uint32_t *)f.col)[row];
      if (x >= f.ncat) continue;
      if (f.family == FAM_BB) {  // ss = [heads, tails]
        const int j = x ? 0 : 1;
        if (a >= 0) atomic_add_f64(blk + (size_t)a * 2 + j, -1.0);
        if (b >= 0) atomic_add_f64(blk + (size_t)b * 2 + j, 1.0);
      } else if (f.family == FAM_BBNC) {  // ss = [p, heads, tails]: p is the group's parameter, never a delta
        const int j = x ? 1 : 2;
        if (a >= 0) atomic_add_f64(blk + (size_t)a * 3 + j, -1.0);
        if (b >= 0) atomic_add_f64(blk + (size_t)b * 3 + j, 1.0);
      } else {  // ss = [count_sum, counts[dim]]; count_sum is re-derived from counts (dd_count_sum_kernel):
                // a RED per cell on only K addresses per feature would serialise in L2
        if (a >= 0) atomic_add_f64(blk + (size_t)a * f.ss_w + 1 + x, -1.0);
        if (b >= 0) atomic_add_f64(blk + (size_t)b * f.ss_w + 1 + x, 1.0);
      }
    } else if (f.kind == KIND_GP) {  // ss = [count, sum, log_prod]
      const uint32_t x = ((const uint32_t *)f.col)[row];
      if (x == GP_SENTINEL) continue;
      if (f.family == FAM_BNB) {  // ss = [count, sum]
        const double xb = (double)x;
        if (a >= 0) { double *p = blk + (size_t)a * 2; atomic_add_f64(p, -1.0); atomic_add_f64(p + 1, -xb); }
        if (b >= 0) { double *p = blk + (size_t)b * 2; atomic_add_f64(p, 1.0); atomic_add_f64(p + 1, xb); }
        continue;
      }
      const double xd = (double)x, lf = lgamma(xd + 1.0);
      if (a >= 0) { double *p = blk + (size_t)a * 3; atomic_add_f64(p, -1.0); atomic_add_f64(p + 1, -xd); atomic_add_f64(p + 2, -lf); }
      if (b >= 0) { double *p = blk + (size_t)b * 3; atomic_add_f64(p, 1.0); atomic_add_f64(p + 1, xd); atomic_add_f64(p + 2, lf); }
    } else if (f.kind == KIND_NICH) {  // ss = [count, sum x, sum x^2]
      const float xf = ((const float *)f.col)[row];
      if (xf != xf) continue;
      const double xd = (double)xf, x2 = xd * xd;
      if (a >= 0) { double *p = blk + (size_t)a * 3; atomic_add_f64(p, -1.0); atomic_add_f64(p + 1, -xd); atomic_add_f64(p + 2, -x2); }
      if (b >= 0) { double *p = blk + (size_t)b * 3; atomic_add_f64(p, 1.0); atomic_add_f64(p + 1, xd); atomic_add_f64(p + 2, x2); }
    }
  }
}

// NIW update: one warp per moved row, lanes over the d + d*d moment entries.
__global__ void update_niw_kernel(FeatDev f, const int32_t *__restrict__ old_slot, const int32_t *__restrict__ new_slot,
                                  size_t row_lo, size_t row_hi, double *__restrict__ delta) {
  const size_t row = row_lo + (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= row_hi) return;
  const int a = old_slot ? old_slot[row] : -1;
  const int b = new_slot ? new_slot[row - row_lo] : -1;
  if (a == b) return;
  const int d = (int)f.dim;
  const float *x = (const float *)f.col + row * (size_t)d;
  if (x[0] != x[0]) return;
  double *blk = delta + f.ss_off;
  if (lane == 0) {
    if (a >= 0) atomic_add_f64(blk + (size_t)a * f.ss_w, -1.0);
    if (b >= 0) atomic_add_f64(blk + (size_t)b * f.ss_w, 1.0);
  }
  for (int e = lane; e < d + d * d; e += 32) {
    double v;
    if (e < d) v = (double)x[e];
    else { const int i = (e - d) / d, j = (e - d) - i * d; v = (double)x[i] * (double)x[j]; }
    if (a >= 0) atomic_add_f64(blk + (size_t)a * f.ss_w + 1 + e, -v);
    if (b >= 0) atomic_add_f64(blk + (size_t)b * f.ss_w + 1 + e, v);
  }
}

// CRP bookkeeping (group_manager.hpp:218-248): per-group entity counts,
// assignment vector, number of moved rows.
__global__ void commit_assign_kernel(int32_t *__restrict__ assign, const int32_t *__restrict__ new_slot,
                                     size_t row_lo, size_t row_hi, double *__restrict__ delta_counts, int kmax,
                                     unsigned long long *__restrict__ moved) {
  // per-block histogram of count changes in shared memory (when it fits), one RED per touched group per block
  extern __shared__ int hist[];
  const bool use_hist = kmax <= 8192;
  if (use_hist) {
    for (int i = threadIdx.x; i < kmax; i += blockDim.x) hist[i] = 0;
    __syncthreads();
  }
  const size_t row = row_lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool did = false;
  if (row < row_hi) {
    const int a = assign[row], b = new_slot[row - row_lo];
    if (a != b) {
      if (use_hist) {
        if (a >= 0) atomicSub(&hist[a], 1);
        if (b >= 0) atomicAdd(&hist[b], 1);
      } else {
        if (a >= 0) atomic_add_f64(delta_counts + a, -1.0);
        if (b >= 0) atomic_add_f64(delta_counts + b, 1.0);
      }
      assign[row] = b;
      did = true;
    }
  }
  const unsigned m = __ballot_sync(0xffffffffu, did);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(moved, (unsigned long long)__popc(m));
  if (use_hist) {
    __syncthreads();
    for (int i = threadIdx.x; i < kmax; i += blockDim.x)
      if (hist[i] != 0) atomic_add_f64(delta_counts + i, (double)hist[i]);
  }
}

// dd: count_sum[slot] = sum of counts[slot][:] (kept consistent after every apply)
__global__ void dd_count_sum_kernel(const FeatDev *__restrict__ feats, int nfeat, int kmax, double *__restrict__ ss) {
  const int d = blockIdx.y;
  const FeatDev f = feats[d];
  if (f.family != FAM_DD) return;
  const int slot = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (slot >= kmax) return;
  double *p = ss + f.ss_off + (size_t)slot * f.ss_w;
  double s = 0.0;
  for (uint32_t i = lane; i < f.dim; i += 32) s += p[1 + i];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) p[0] = s;
}

// count-valued states (bb / dd only): the deltas are numbers of rows, exact in int32 -- half the bytes of the fp64 buffer
__global__ void delta_to_i32_kernel(const double *__restrict__ delta, size_t n, int32_t *__restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int32_t)delta[i];
}
__global__ void delta_from_i32_kernel(const int32_t *__restrict__ in, size_t n, double *__restrict__ delta) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) delta[i] = (double)in[i];
}

__global__ void apply_delta_kernel(double *__restrict__ ss, double *__restrict__ delta, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { ss[i] += delta[i]; delta[i] = 0.0; }
}

// base[c] = log(pseudocount(group of column c)) (group_manager.hpp:274-283): the group's entity count, or
// alpha / #empty groups for an empty one; columns [ncols, ld) are padding (-inf).  Computed on the device from
// the resident counts so that a sweep never needs the host copy.  One block.
__global__ void base_kernel(const double *__restrict__ counts, const int32_t *__restrict__ col2slot, int ncols, int ld,
                            float alpha, float *__restrict__ base) {
  __shared__ int s_empty;
  if (threadIdx.x == 0) s_empty = 0;
  __syncthreads();
  int e = 0;
  for (int c = threadIdx.x; c < ncols; c += blockDim.x) e += counts[col2slot[c]] == 0.0;
  for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
  if ((threadIdx.x & 31) == 0 && e) atomicAdd(&s_empty, e);
  __syncthreads();
  const float per_empty = __fdiv_rn(alpha, (float)s_empty);
  for (int c = threadIdx.x; c < ld; c += blockDim.x) {
    float v = -CUDART_INF_F;
    if (c < ncols) {
      const double cnt = counts[col2slot[c]];
      v = (float)log((double)(cnt != 0.0 ? (float)cnt : per_empty));
    }
    base[c] = v;
  }
}

// base[col] += sum over nich features of c0[col] (and over binary-form bb features of t0[col]): the row-independent
// part of the term is added once per (row, group) in the score kernel's epilogue instead of once per unit
__global__ void nich_c0_sum_kernel(const FeatDev *__restrict__ feats, int nfeat, const float *__restrict__ params,
                                   size_t region_rows, int KT, int ncols_padded, float *__restrict__ base) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncols_padded) return;
  const int kt = col / KT, kl = col - kt * KT;
  float s = 0.f;
  for (int d = 0; d < nfeat; d++) {
    const FeatDev f = feats[d];
    if (f.kind == KIND_TABLE && f.binform) s += params[((size_t)kt * region_rows + f.rowoff + 1) * KT + kl];  // t0
    if (f.kind != KIND_NICH) continue;
    s += params[((size_t)kt * region_rows + f.rowoff + 3) * KT + kl];
  }
  base[col] += s;
}

// scores[r][c] = base[c]: the CRP term, when no scalar feature kernel initialises the matrix
// Small copies that stay OFF the copy engines: a cudaMemcpyAsync -- device to device included -- queues on a DMA engine
// behind whatever that engine is moving, and on a pass over host rows that is the next pass's 32 MB of records: with
// eight GPUs uploading at once the sweep's "build" phase waited 0.3 ms for a 1 KB copy (bench.py, device_phase_ms_per_pass).
__global__ void copy_f32_kernel(const float *__restrict__ src, float *__restrict__ dst, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}
__global__ void zero_u64_kernel(unsigned long long *p) { *p = 0ull; }
// the moved-row counter straight into (mapped, pinned) host memory
__global__ void publish_counter_kernel(const unsigned long long *__restrict__ d, unsigned long long *__restrict__ h) {
  *h = *d;
  __threadfence_system();
}
__global__ void fill_rows_kernel(float *__restrict__ scores, size_t ld, const float *__restrict__ base, size_t nrows) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nrows * ld) scores[i] = base[i % ld];
}

// gid <-> slot translation of the assignment vector
__global__ void map_i32_to_i64_kernel(const int32_t *__restrict__ in, const int64_t *__restrict__ table, size_t n,
                                      int64_t *__restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i] < 0 ? -1 : table[in[i]];
}

// ---------------------------------------------------------------------------
// Single-value plugin calls (models/base.hpp:25-27) on the device.  ss here is
// the reference's field representation (nich: count, mean, count_times_variance).
// op: 0 score, 1 add, 2 remove.
// ---------------------------------------------------------------------------
__global__ void value_op_kernel(int family, uint32_t dim, int op, const double *__restrict__ hp, double *__restrict__ ss,
                                const double *__restrict__ x, float *__restrict__ score) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double sgn = op == 2 ? -1.0 : 1.0;
  if (family == FAM_BB) {
    if (op == 0) *score = (float)bb_score(hp, ss, x[0] != 0.0);
    else ss[x[0] != 0.0 ? 0 : 1] += sgn;
  } else if (family == FAM_BBNC) {
    if (op == 0) *score = (float)bbnc_score(ss, x[0] != 0.0);
    else ss[x[0] != 0.0 ? 1 : 2] += sgn;
  } else if (family == FAM_DD) {
    const uint32_t xi = (uint32_t)x[0];
    if (op == 0) {
      double asum = 0.0;
      for (uint32_t i = 0; i < dim; i++) asum += hp[i];
      *score = xi < dim ? (float)dd_score(hp, asum, ss, xi) : CUDART_NAN_F;
    } else if (xi < dim) { ss[0] += sgn; ss[1 + xi] += sgn; }
  } else if (family == FAM_BNB) {
    if (op == 0) *score = (float)bnb_score(bnb_post(hp, ss), x[0]);
    else { ss[0] += sgn; ss[1] += sgn * x[0]; }
  } else if (family == FAM_GP) {
    if (op == 0) *score = (float)gp_score(gp_post(hp, ss), x[0]);
    else { ss[0] += sgn; ss[1] += sgn * x[0]; ss[2] += sgn * lgamma(x[0] + 1.0); }
  } else if (family == FAM_NICH) {
    double add[3] = {ss[0], ss[0] * ss[1], ss[2] + ss[0] * ss[1] * ss[1]};  // -> (n, sum x, sum x^2)
    if (op == 0) *score = (float)nich_score(nich_post(hp, add), x[0]);
    else {
      add[0] += sgn; add[1] += sgn * x[0]; add[2] += sgn * x[0] * x[0];
      ss[0] = add[0];
      ss[1] = add[0] > 0.0 ? add[1] / add[0] : 0.0;
      double ctv = add[0] > 1.0 ? add[2] - add[1] * ss[1] : 0.0;
      ss[2] = ctv > 0.0 ? ctv : 0.0;
    }
  } else if (family == FAM_DM) {  // ss = [counts[dim], ratio]; x = dim counts
    double X = 0.0, part = 0.0;
    for (uint32_t i = 0; i < dim; i++) { X += x[i]; part += lgamma(x[i] + 1.0); }
    if (op == 0) {
      double s = lgamma(X + 1.0) - part, E = 0.0;
      for (uint32_t i = 0; i < dim; i++) { const double e = hp[i] + ss[i]; E += e; s += lgamma_rise(e, (uint32_t)x[i]); }
      *score = (float)(s + lgamma(E) - lgamma(E + X));
    } else {
      for (uint32_t i = 0; i < dim; i++) ss[i] += sgn * x[i];
      ss[dim] += sgn * (lgamma(X + 1.0) - part);
    }
  } else if (family == FAM_NIW && op != 0) {
    ss[0] += sgn;
    for (uint32_t i = 0; i < dim; i++) ss[1 + i] += sgn * x[i];
    for (uint32_t i = 0; i < dim; i++)
      for (uint32_t j = 0; j < dim; j++) ss[1 + dim + i * dim + j] += sgn * x[i] * x[j];
  }
}

}  // namespace msb
