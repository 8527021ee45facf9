// Non-conjugate parameters on the device (DESIGN.md section 4.11): the mixturemodel runner's theta kernel -- one
// univariate slice-sampling update (Neal 2003: stepping out, then shrinkage) of every group's bbnc p -- and the
// auxiliary-parameter step of Neal's algorithm 8, a fresh p ~ Beta(alpha, beta) for every empty group.
//
// One thread per (feature, group column): a chain reads p, heads and tails.  Each column draws from its own Philox
// stream, keyed by the group id rather than the slot, and nothing is summed across columns, so replicas with identical
// suffstats draw identical p without a collective.  Block b of the stream of (feature d, gid g, call counter c) is
// philox4x32_10(key = seed, counter = (c << 32 | g, TAG | d << 16 | b)): g < 2^32, c < 2^32, d < 2^16, and b < 2^16
// (a slice update reads at most 1 + THETA_SHRINK_CAP / 2 blocks, a Beta draw at most ~3000).
//
// The kernels write to scratch (p, and a status per column); the host commits with theta_commit_kernel only once it
// has seen that no column was refused.
#pragma once
#include "msb_draw.cuh"

namespace msb {

constexpr uint64_t THETA_TAG = 0x534c494300000000ull;  // "SLIC": the slice updates' counters, apart from the sweeps',
constexpr uint64_t AUX_TAG = 0x4155585000000000ull;    // "AUXP": DRAW_TAG's, HP_TAG's and the group_seed stream's
constexpr int THETA_SHRINK_CAP = 200;                   // shrink steps of one update; a column that reaches it keeps p0
constexpr uint32_t THETA_STEP_CAP = 1u << 20;           // stepping-out steps per side (w >= 1e-6 covers [0, 1])
constexpr int THETA_THREADS = 128;

enum ThetaStatus : uint8_t { THETA_NEW = 0, THETA_CAPPED = 1, THETA_BAD = 2, THETA_KEEP = 3 };

// one feature a launch covers (blockIdx.y); w = the slice width (theta_kernel only)
struct ThetaFeat { int32_t feat; uint32_t pad; double w; };

// the bbnc density of group::score_data (score_data_cell) at p, for the group's heads and tails
__device__ __forceinline__ double bbnc_target(const FeatDev &f, const double *__restrict__ h, double p, double heads, double tails) {
  const double g[3] = {p, heads, tails};
  return score_data_cell(f, h, f.asum, g);
}

// flags[0] += columns that reached a cap, flags[1] = min over refused columns of (launch row * ncols + column)
__device__ __forceinline__ void theta_flag(uint32_t *flags, uint8_t s, uint32_t o) {
  if (s == THETA_CAPPED) atomicAdd(&flags[0], 1u);
  else if (s == THETA_BAD) atomicMin(&flags[1], o);
}

// One slice update per (feature tf[blockIdx.y], column).  y = f(p0) + log u with u = (i + 1/2) 2^-52 strictly inside
// (0, 1); L = p0 - w u', R = L + w, stepped out by w while f > y; then x = L + u'' (R - L) until f(x) > y, shrinking the
// side of p0 that x fell on.  NaN compares false: outside the slice.  The products and sums are rounded one by one
// (no FMA contraction) so that a restatement in plain fp64 reproduces them.
__global__ void __launch_bounds__(THETA_THREADS) theta_kernel(const FeatDev *__restrict__ feats, const ThetaFeat *__restrict__ tf,
                                                              const double *__restrict__ hp, const double *__restrict__ ss,
                                                              const int32_t *__restrict__ col2slot, const uint32_t *__restrict__ colgid,
                                                              int ncols, uint64_t seed, uint64_t counter, double *__restrict__ pnew,
                                                              uint8_t *__restrict__ status, uint32_t *__restrict__ flags) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncols) return;
  const ThetaFeat t = tf[blockIdx.y];
  const FeatDev f = feats[t.feat];
  const double *h = hp + f.hp_off;
  const double *g = ss + f.ss_off + (size_t)col2slot[c] * f.ss_w;
  const double p0 = g[0], heads = g[1], tails = g[2], w = t.w;
  const uint32_t o = blockIdx.y * (uint32_t)ncols + (uint32_t)c;
  const double f0 = bbnc_target(f, h, p0, heads, tails);
  uint8_t s = THETA_CAPPED;
  double p = p0;
  if (!isfinite(f0)) {
    s = THETA_BAD;
  } else {
    DrawStream rs(seed, counter << 32 | colgid[c], THETA_TAG | (uint64_t)t.feat << 16);
    const uint32_t a = rs.next() >> 6, b = rs.next() >> 6;
    const double y = f0 + log(((double)a * 67108864.0 + (double)b + 0.5) * (1.0 / 4503599627370496.0));
    double L = __dsub_rn(p0, __dmul_rn(w, rs.u53()));
    double R = __dadd_rn(L, w);
    uint32_t n = 0;
    while (n <= THETA_STEP_CAP && bbnc_target(f, h, L, heads, tails) > y) { L = __dsub_rn(L, w); n++; }
    uint32_t m = 0;
    while (m <= THETA_STEP_CAP && bbnc_target(f, h, R, heads, tails) > y) { R = __dadd_rn(R, w); m++; }
    if (n <= THETA_STEP_CAP && m <= THETA_STEP_CAP) {
      for (int i = 0; i < THETA_SHRINK_CAP; i++) {
        const double x = __dadd_rn(L, __dmul_rn(rs.u53(), __dsub_rn(R, L)));
        if (bbnc_target(f, h, x, heads, tails) > y) { p = x; s = THETA_NEW; break; }
        if (x < p0) L = x;
        else R = x;
      }
    }
  }
  pnew[o] = p;
  status[o] = s;
  theta_flag(flags, s, o);
}

// Algorithm 8's auxiliary parameters: every column of feature tf[blockIdx.y] whose resident count is 0 gets
// p = x / (x + y), x ~ Gamma(alpha), y ~ Gamma(beta) (DrawStream::gamma, in that order); a column with members is kept.
// A draw that is not in [0, 1] (both gammas underflowed) is refused.
__global__ void __launch_bounds__(THETA_THREADS) redraw_empty_kernel(const FeatDev *__restrict__ feats, const ThetaFeat *__restrict__ tf,
                                                                     const double *__restrict__ hp, const double *__restrict__ ss,
                                                                     const int32_t *__restrict__ col2slot, const uint32_t *__restrict__ colgid,
                                                                     int ncols, uint64_t seed, uint64_t counter, double *__restrict__ pnew,
                                                                     uint8_t *__restrict__ status, uint32_t *__restrict__ flags) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncols) return;
  const ThetaFeat t = tf[blockIdx.y];
  const uint32_t o = blockIdx.y * (uint32_t)ncols + (uint32_t)c;
  const int slot = col2slot[c];
  if (ss[slot] != 0.0) { status[o] = THETA_KEEP; return; }  // d_ss[0, kmax) holds the entity counts
  const FeatDev f = feats[t.feat];
  const double *h = hp + f.hp_off;
  DrawStream rs(seed, counter << 32 | colgid[c], AUX_TAG | (uint64_t)t.feat << 16);
  const double x = rs.gamma(h[0]);
  const double y = rs.gamma(h[1]);
  const double p = x / (x + y);
  const uint8_t s = (p >= 0.0 && p <= 1.0) ? THETA_NEW : THETA_BAD;
  pnew[o] = p;
  status[o] = s;
  theta_flag(flags, s, o);
}

// the commit: p of every THETA_NEW column into the resident suffstats
__global__ void theta_commit_kernel(const FeatDev *__restrict__ feats, const ThetaFeat *__restrict__ tf,
                                    const int32_t *__restrict__ col2slot, int ncols, const double *__restrict__ pnew,
                                    const uint8_t *__restrict__ status, double *__restrict__ ss) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncols) return;
  const uint32_t o = blockIdx.y * (uint32_t)ncols + (uint32_t)c;
  if (status[o] != THETA_NEW) return;
  const FeatDev f = feats[tf[blockIdx.y].feat];
  ss[f.ss_off + (size_t)col2slot[c] * f.ss_w] = pnew[o];
}

}  // namespace msb
