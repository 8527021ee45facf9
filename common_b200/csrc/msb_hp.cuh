// Hyperparameter inference on a grid (msb_state_hp_gibbs, DESIGN.md section 4.10): one Gibbs step for every feature
// that has a grid of hp vectors and for the CRP concentration alpha if it has one.
//
// For a feature d and a grid point theta_g the weight is L_d[g] = sum over every group column c (ascending gid order,
// empty groups included) of group::score_data(c, d; theta_g) in fp64, the same closed forms score_data_kernel
// evaluates (score_data_cell, niw below).  For alpha: L[g] = (#non-empty - 1) log alpha_g + lgamma(1 + alpha_g) -
// lgamma(n + alpha_g), the alpha-dependent part of score_assignment_kernel's closed form.
//
// Every sum over groups has a fixed order -- per-thread partials over a strided column range, a fixed shuffle tree
// inside the warp, the warp partials added in warp order by thread 0 -- and there are no floating-point atomics, so
// bit-identical suffstats give bit-identical weights and draws (the replicas of a row-sharded run draw the same hypers
// without a collective).
#pragma once
#include "msb_kernels.cuh"

namespace msb {

constexpr uint64_t HP_TAG = 0x4859505200000000ull;  // "HYPR": keeps these counters apart from the sweeps', DRAW_TAG's and
                                                    // the bbnc group streams'
constexpr int HP_THREADS = 128;

// one grid: a feature's (feat < nfeat) or alpha's (feat == nfeat); feat is also the Philox row of the draw
struct HpRow {
  int32_t feat;
  int32_t npoints;
  uint32_t nhp;        // doubles per point (1 for alpha)
  uint32_t pad;
  uint64_t pt_off;     // points[pt_off + g * nhp + j]
  uint64_t lp_off;     // log_prior[lp_off + g]
};

// the block's sum of one value per thread, in a fixed order; the result is valid in thread 0
__device__ __forceinline__ double hp_block_sum(double v) {
  __shared__ double s_part[HP_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += s_part[w];
  return s;
}

// every family but niw: one block per (grid row, grid point), threads over the group columns.
// L[row * ld + g] = sum_c score_data_cell(theta_g, column c)
__global__ void __launch_bounds__(HP_THREADS, 2) hp_grid_kernel(const FeatDev *__restrict__ feats, int nfeat,
                                                                const HpRow *__restrict__ rows, const double *__restrict__ pts,
                                                                const double *__restrict__ ss, const int32_t *__restrict__ col2slot,
                                                                int ncols, size_t ld, double *__restrict__ L) {
  const HpRow row = rows[blockIdx.x];
  const int g = blockIdx.y;
  if (row.feat >= nfeat || g >= row.npoints) return;
  const FeatDev f = feats[row.feat];
  if (f.kind == KIND_NIW) return;  // niw_hp_* below
  const double *h = pts + row.pt_off + (size_t)g * row.nhp;
  double asum = 0.0;  // dd: summed in the order msb_state_set_hp sums it
  if (f.family == FAM_DD)
    for (uint32_t c = 0; c < f.dim; c++) asum += h[c];
  double s = 0.0;
  for (int c = threadIdx.x; c < ncols; c += blockDim.x)
    s += score_data_cell(f, h, asum, ss + f.ss_off + (size_t)col2slot[c] * f.ss_w);
  s = hp_block_sum(s);
  if (threadIdx.x == 0) L[blockIdx.x * ld + g] = s;
}

// niw, the group-independent prior term: ld0[g] = log |psi0_g|, one block per grid point
__global__ void niw_hp_prior_kernel(int d, const double *__restrict__ pts, uint32_t nhp, double *__restrict__ ld0) {
  extern __shared__ double sm[];
  __shared__ int s_fail;
  __shared__ double s_acc;
  const double *psi0 = pts + (size_t)blockIdx.x * nhp + d + 1;
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) sm[e] = psi0[e];
  __syncthreads();
  const double ld = block_chol_logdet(sm, d, &s_fail, &s_acc);
  if (threadIdx.x == 0) ld0[blockIdx.x] = ld;
}

// niw, one block per (group column, grid point): niw_score_data_kernel's closed form with the prior's log |psi0| from
// niw_hp_prior_kernel.  out[g * ncols + col]
__global__ void niw_hp_group_kernel(FeatDev f, const double *__restrict__ pts, uint32_t nhp, const double *__restrict__ ld0,
                                    const double *__restrict__ ss, const int32_t *__restrict__ col2slot, int ncols,
                                    double *__restrict__ out) {
  extern __shared__ double sm[];
  const int d = (int)f.dim;
  double *A = sm;          // d*d
  double *mu = A + d * d;  // d
  __shared__ int s_fail;
  __shared__ double s_acc;
  const int k = blockIdx.x, g = blockIdx.y;
  const double *fhp = pts + (size_t)g * nhp;
  const double *gss = ss + f.ss_off + (size_t)col2slot[k] * f.ss_w;
  const double *mu0 = fhp, kappa0 = fhp[d], *psi0 = fhp + d + 1, nu0 = fhp[d + 1 + (size_t)d * d];
  const double n = gss[0];
  const double *sx = gss + 1, *sxx = gss + 1 + d;
  const double kn = kappa0 + n, nun = nu0 + n;
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
    out[(size_t)g * ncols + k] = -0.5 * n * d * log(CUDART_PI) + lg + 0.5 * nu0 * ld0[g] - 0.5 * nun * ldn +
                                 0.5 * d * log(kappa0 / kn);
  }
}

// niw, the second pass: L[g] = sum over the columns of in[g * ncols + c], one block per grid point
__global__ void __launch_bounds__(HP_THREADS) hp_reduce_kernel(const double *__restrict__ in, int ncols, double *__restrict__ L) {
  double s = 0.0;
  for (int c = threadIdx.x; c < ncols; c += blockDim.x) s += in[(size_t)blockIdx.x * ncols + c];
  s = hp_block_sum(s);
  if (threadIdx.x == 0) L[blockIdx.x] = s;
}

// alpha: one block over the resident counts
__global__ void __launch_bounds__(HP_THREADS) hp_alpha_kernel(const double *__restrict__ counts, const int32_t *__restrict__ col2slot,
                                                              int ncols, const double *__restrict__ alphas, int npoints,
                                                              double *__restrict__ L) {
  __shared__ double s_ne, s_n;
  double ne = 0.0, n = 0.0;
  for (int c = threadIdx.x; c < ncols; c += blockDim.x) {
    const double cnt = counts[col2slot[c]];
    if (cnt > 0.0) { ne += 1.0; n += cnt; }
  }
  ne = hp_block_sum(ne);
  __syncthreads();  // hp_block_sum's partials are read before they are reused
  n = hp_block_sum(n);
  if (threadIdx.x == 0) { s_ne = ne; s_n = n; }
  __syncthreads();
  for (int g = threadIdx.x; g < npoints; g += blockDim.x) {
    const double a = alphas[g];
    L[g] = (s_ne - 1.0) * log(a) + lgamma(1.0 + a) - lgamma(s_n + a);
  }
}

// one thread per grid: w_g = log_prior[g] + L[g] into logw, m = max w, p_g = exp(w_g - m) summed in index order in
// fp64, choice = the first g whose running sum exceeds u * sum p, u = a 53-bit uniform from philox4x32_10(seed, row,
// HP_TAG | counter) built as DrawStream::u53 builds it.  A NaN or +inf weight, or a grid of -inf weights: choice -1
// (the host reads logw to say which).
__global__ void hp_draw_kernel(const HpRow *__restrict__ rows, int nrows, const double *__restrict__ log_prior,
                               const double *__restrict__ L, size_t ld, uint64_t seed, uint64_t counter,
                               double *__restrict__ logw, int64_t *__restrict__ choice) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nrows) return;
  const HpRow row = rows[r];
  const double *w = logw + r * ld;
  double m = -CUDART_INF;
  bool nan = false;
  for (int g = 0; g < row.npoints; g++) {
    const double v = log_prior[row.lp_off + g] + L[r * ld + g];
    logw[r * ld + g] = v;
    if (isnan(v) || v == CUDART_INF) nan = true;
    else if (v > m) m = v;
  }
  if (nan || m == -CUDART_INF) { choice[r] = -1; return; }
  double tot = 0.0;
  for (int g = 0; g < row.npoints; g++) tot += exp(w[g] - m);
  uint32_t q[4];
  philox4x32_10(seed, (uint64_t)row.feat, HP_TAG | counter, q);
  const double u = ((double)(q[0] >> 5) * 67108864.0 + (double)(q[1] >> 6)) * (1.0 / 9007199254740992.0);
  const double t = u * tot;
  double acc = 0.0;
  int pick = -1;
  for (int g = 0; g < row.npoints; g++) {
    const double p = exp(w[g] - m);
    acc += p;
    if (p > 0.0) pick = g;  // the last point with p > 0: where u * tot rounds up to tot
    if (acc > t) { pick = g; break; }
  }
  choice[r] = pick;
}

}  // namespace msb
