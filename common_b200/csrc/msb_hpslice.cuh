// Slice sampling of continuous hypers (msb_state_slice_hp, DESIGN.md section 4.12): the mixturemodel runner's slice hp
// kernel -- one univariate slice update (Neal 2003: bounded stepping out, then shrinkage) per (feature, scalar hp key),
// and of the CRP concentration alpha.
//
// The target of coordinate x of feature d is f(x) = log prior(x) + sum over every group column c (ascending gid order,
// empty groups included, the set hp_gibbs sums) of score_data_cell(c, d; theta with x substituted), in fp64 with
// hp_block_sum's fixed order and no atomics; -inf outside the key's support.  alpha's is log prior(x) + (#non-empty - 1)
// log x + lgamma(1 + x) - lgamma(n + x), hp_alpha_kernel's closed form.  niw evaluates the rank-one form
//   log |psi'_c| = log |B_c| + log1p(kappa n_c q_c / (kappa + n_c)),  B_c = psi + sum xx^T - sum x sum x^T / n_c,
//   q_c = v^T B_c^-1 v,  v = mean_c - mu0
// from niw_slice_prep_kernel, so an evaluation costs O(K d) instead of K Cholesky factorisations.
//
// One block per feature (and one for alpha): its specs run in the order given, each conditioning on the values its
// predecessors drew.  Every thread of the block runs the same slice arithmetic on the same stream and sees the same
// block-wide f, so every loop is block-uniform.  Spec j of feature d (alpha: d = nfeat) reads Philox block b of
// philox4x32_10(key = seed, counter = (counter << 32 | d, HPSL_TAG | j << 16 | b)); an update reads at most about 103
// blocks.  Identical suffstats and hypers give identical bits, so row-sharded replicas draw the same hypers without a
// collective.  The kernel writes the new values and a status per spec to scratch; the host commits them.
#pragma once
#include "msb_draw.cuh"
#include "msb_hp.cuh"

namespace msb {

constexpr uint64_t HPSL_TAG = 0x4850534c00000000ull;  // "HPSL": apart from the sweeps', DRAW_TAG's, HP_TAG's, THETA_TAG's
constexpr int HPSL_STEP_M = 128;                       // Neal's m: at most m - 1 stepping-out steps over both sides
constexpr int HPSL_SHRINK_CAP = 200;                   // shrink steps of one update; a spec that reaches it keeps x0

enum HpPrior : int32_t { HPRIOR_FLAT = 0, HPRIOR_EXPONENTIAL = 1, HPRIOR_NORMAL = 2, HPRIOR_NONINFORMATIVE_BETA = 3 };
enum HpSliceStatus : uint8_t { HPSL_NEW = 0, HPSL_CAPPED = 1, HPSL_BAD = 2 };

// one coordinate to update
struct HpSliceSpec {
  int32_t slot;     // the coordinate in HpSliceFeat::h
  int32_t partner;  // HPRIOR_NONINFORMATIVE_BETA: the slot of the other of (alpha, beta)
  int32_t prior;    // HpPrior
  uint32_t out;     // the spec's index in the caller's array
  double w, a, b;   // width, prior parameters
  double lo;        // the support is x > lo (-inf: the real line)
};

// one block: a feature (feat < nfeat) or alpha (feat == nfeat) and its specs[first, first + nspecs)
struct HpSliceFeat {
  int32_t feat;
  int32_t niw;      // niw: the row of the prep scratch; -1 otherwise
  uint32_t first, nspecs;
  double h[4];      // current values: the family's hp vector (<= 4 scalars); niw: kappa, nu; alpha: alpha
};

__device__ __forceinline__ double hpsl_log_prior(const HpSliceSpec &s, double x, const double *h) {
  switch (s.prior) {
    case HPRIOR_FLAT: return (x > s.a && x < s.b) ? 0.0 : -CUDART_INF;
    case HPRIOR_EXPONENTIAL: return x >= 0.0 ? __dsub_rn(log(s.a), __dmul_rn(s.a, x)) : -CUDART_INF;
    case HPRIOR_NORMAL: {
      const double t = __dsub_rn(x, s.a);
      return __dsub_rn(__dmul_rn(-0.5, log(__dmul_rn(6.283185307179586, s.b))), __ddiv_rn(__dmul_rn(t, t), __dmul_rn(2.0, s.b)));
    }
    default: return __dmul_rn(-2.5, log(__dadd_rn(x, h[s.partner])));  // -2.5 log(alpha + beta)
  }
}

// niw's score_data of one column at (kappa, nu) from the prep values (n, log |B|, q) and ld0 = log |psi|
__device__ __forceinline__ double niw_slice_cell(int d, double kappa, double nu, const double *__restrict__ p, double ld0) {
  const double n = p[0];
  if (n == 0.0) return 0.0;
  const double kn = kappa + n, nun = nu + n;
  double lg = 0.0;  // lgamma_d(nu'/2) - lgamma_d(nu/2): the pi^(d(d-1)/4) factors cancel
  for (int j = 0; j < d; j++) lg += lgamma(0.5 * (nun - j)) - lgamma(0.5 * (nu - j));
  const double ldn = p[1] + log1p(kappa * n * p[2] / kn);
  return -0.5 * n * d * log(CUDART_PI) + lg + 0.5 * nu * ld0 - 0.5 * nun * ldn + 0.5 * d * log(kappa / kn);
}

// niw, once per call and feature: one block per group column c < ncols writes prep[c * 3 + {0, 1, 2}] = (n_c, log |B_c|,
// q_c), (0, 0, 0) for an empty group; block ncols writes *ld0 = log |psi|.  Shared: B [d * d] | v [d]
__global__ void niw_slice_prep_kernel(FeatDev f, const double *__restrict__ hp, const double *__restrict__ ss,
                                      const int32_t *__restrict__ col2slot, int ncols, double *__restrict__ prep,
                                      double *__restrict__ ld0) {
  extern __shared__ double sm[];
  __shared__ int s_fail;
  __shared__ double s_acc;
  const int d = (int)f.dim, k = blockIdx.x;
  double *A = sm, *v = A + d * d;
  const double *mu0 = hp + f.hp_off, *psi0 = mu0 + d + 1;
  if (k == ncols) {
    for (int e = threadIdx.x; e < d * d; e += blockDim.x) A[e] = psi0[e];
    __syncthreads();
    const double ld = block_chol_logdet(A, d, &s_fail, &s_acc);
    if (threadIdx.x == 0) *ld0 = ld;
    return;
  }
  const double *gss = ss + f.ss_off + (size_t)col2slot[k] * f.ss_w;
  const double n = gss[0];
  double *out = prep + (size_t)k * 3;
  if (n == 0.0) {
    if (threadIdx.x == 0) { out[0] = 0.0; out[1] = 0.0; out[2] = 0.0; }
    return;
  }
  const double *sx = gss + 1, *sxx = gss + 1 + d;
  for (int i = threadIdx.x; i < d; i += blockDim.x) v[i] = sx[i] / n - mu0[i];
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) {
    const int i = e / d, j = e - i * d;
    A[e] = psi0[e] + sxx[e] - sx[i] * sx[j] / n;
  }
  __syncthreads();
  const double ldB = block_chol_logdet(A, d, &s_fail, &s_acc);  // A's lower triangle is now L, L L^T = B
  if (threadIdx.x == 0) {
    double q = 0.0;  // |L^-1 v|^2 by forward substitution, z overwriting v
    for (int i = 0; i < d; i++) {
      double t = v[i];
      for (int m = 0; m < i; m++) t -= A[i * d + m] * v[m];
      v[i] = t / A[i * d + i];
      q += v[i] * v[i];
    }
    out[0] = n; out[1] = ldB; out[2] = q;
  }
}

// Block-wide f(x) for spec s: every thread calls it with the same x and gets the same value.  The coordinate is
// written to s_h[s.slot] (the caller restores it); a prior or support of -inf skips the sum.
__device__ __forceinline__ double hpsl_target(const HpSliceFeat &t, const HpSliceSpec &s, const FeatDev &f, bool is_alpha, double x,
                              double *s_h, double *s_f, double ne, double n, const double *__restrict__ ss,
                              const int32_t *__restrict__ col2slot, int ncols, const double *__restrict__ prep, double ld0) {
  __syncthreads();  // the previous evaluation's readers of s_h and s_f are done
  const double lp = x > s.lo ? hpsl_log_prior(s, x, s_h) : -CUDART_INF;
  if (!(lp > -CUDART_INF)) return lp;
  if (is_alpha)
    return __dadd_rn(lp, __dsub_rn(__dadd_rn(__dmul_rn(ne - 1.0, log(x)), lgamma(__dadd_rn(1.0, x))), lgamma(__dadd_rn(n, x))));
  if (threadIdx.x == 0) s_h[s.slot] = x;
  __syncthreads();
  double v = 0.0;
  if (t.niw >= 0) {
    const double kappa = s_h[0], nu = s_h[1];
    for (int c = threadIdx.x; c < ncols; c += blockDim.x) v += niw_slice_cell((int)f.dim, kappa, nu, prep + (size_t)c * 3, ld0);
  } else {
    for (int c = threadIdx.x; c < ncols; c += blockDim.x) v += score_data_cell(f, s_h, f.asum, ss + f.ss_off + (size_t)col2slot[c] * f.ss_w);
  }
  v = hp_block_sum(v);
  if (threadIdx.x == 0) *s_f = __dadd_rn(lp, v);
  __syncthreads();
  return *s_f;
}

// One block per HpSliceFeat.  For each of its specs: y = f(x0) + log u with u = (i + 1/2) 2^-52 strictly inside (0, 1);
// L = x0 - w u', R = L + w; J_L = floor(m V), J_R = m - 1 - J_L; L steps out by w at most J_L times and R at most J_R
// times while f > y (Neal's Fig. 3); then x = L + u'' (R - L) until f(x) > y, shrinking the side of x0 that x fell on.
// NaN compares false: outside the slice.  Products and sums are rounded one by one (no FMA contraction) so that a
// restatement in plain fp64 reproduces them.  val[out] / status[out] per spec; a feature stops at its first HPSL_BAD
// spec (f(x0) not finite), leaving the later specs' status as the host set it.
// One block per feature is few blocks, so the bound asks for registers rather than occupancy: no spills.
__global__ void __launch_bounds__(HP_THREADS, 1) hp_slice_kernel(const FeatDev *__restrict__ feats, int nfeat,
                                                              const HpSliceFeat *__restrict__ tasks,
                                                              const HpSliceSpec *__restrict__ specs, const double *__restrict__ ss,
                                                              const int32_t *__restrict__ col2slot, int ncols,
                                                              const double *__restrict__ niw_prep, const double *__restrict__ niw_ld0,
                                                              uint64_t seed, uint64_t counter, double *__restrict__ val,
                                                              uint8_t *__restrict__ status) {
  __shared__ double s_h[4], s_f, s_ne, s_n;
  const HpSliceFeat t = tasks[blockIdx.x];
  const bool is_alpha = t.feat == nfeat;
  const FeatDev f = feats[is_alpha ? 0 : t.feat];
  const double *prep = t.niw >= 0 ? niw_prep + (size_t)t.niw * ncols * 3 : nullptr;
  const double ld0 = t.niw >= 0 ? niw_ld0[t.niw] : 0.0;
  if (threadIdx.x < 4) s_h[threadIdx.x] = t.h[threadIdx.x];
  if (is_alpha) {  // the counts at d_ss[0, kmax)
    double ne = 0.0, n = 0.0;
    for (int c = threadIdx.x; c < ncols; c += blockDim.x) {
      const double cnt = ss[col2slot[c]];
      if (cnt > 0.0) { ne += 1.0; n += cnt; }
    }
    ne = hp_block_sum(ne);
    __syncthreads();  // hp_block_sum's partials are read before they are reused
    n = hp_block_sum(n);
    if (threadIdx.x == 0) { s_ne = ne; s_n = n; }
  }
  __syncthreads();
  const double ne = is_alpha ? s_ne : 0.0, n = is_alpha ? s_n : 0.0;
  for (uint32_t j = 0; j < t.nspecs; j++) {
    const HpSliceSpec s = specs[t.first + j];
    const double x0 = s_h[s.slot], w = s.w;
    DrawStream rs(seed, counter << 32 | (uint64_t)t.feat, HPSL_TAG | (uint64_t)j << 16);
    uint8_t st = HPSL_CAPPED;
    double x = x0, x1 = x0, y = 0.0, L = 0.0, R = 0.0;
    int phase = 0, jl = 0, jr = 0, shrink = 0;  // phase 0: f(x0), 1: stepping out L, 2: stepping out R, 3: shrinkage
    for (;;) {  // one evaluation per iteration, so that the block-wide target is inlined once
      const double fx = hpsl_target(t, s, f, is_alpha, x, s_h, &s_f, ne, n, ss, col2slot, ncols, prep, ld0);
      if (phase == 0) {
        if (!isfinite(fx)) { st = HPSL_BAD; break; }
        const uint32_t a = rs.next() >> 6, b = rs.next() >> 6;
        y = __dadd_rn(fx, log(((double)a * 67108864.0 + (double)b + 0.5) * (1.0 / 4503599627370496.0)));
        L = __dsub_rn(x0, __dmul_rn(w, rs.u53()));
        R = __dadd_rn(L, w);
        jl = (int)(HPSL_STEP_M * rs.u53());
        jr = HPSL_STEP_M - 1 - jl;
        phase = 1;
      } else if (phase == 1) {
        if (fx > y) { L = __dsub_rn(L, w); jl--; }
        else jl = 0;
      } else if (phase == 2) {
        if (fx > y) { R = __dadd_rn(R, w); jr--; }
        else jr = 0;
      } else {
        if (fx > y) { x1 = x; st = HPSL_NEW; break; }
        if (x < x0) L = x;
        else R = x;
      }
      if (phase == 1 && jl > 0) { x = L; continue; }
      if (phase <= 2) {
        phase = 2;
        if (jr > 0) { x = R; continue; }
        phase = 3;
      }
      if (shrink == HPSL_SHRINK_CAP) break;
      shrink++;
      x = __dadd_rn(L, __dmul_rn(rs.u53(), __dsub_rn(R, L)));
    }
    __syncthreads();
    if (threadIdx.x == 0) { s_h[s.slot] = x1; val[s.out] = x1; status[s.out] = st; }
    __syncthreads();
    if (st == HPSL_BAD) break;
  }
}

}  // namespace msb
