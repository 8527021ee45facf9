// group::sample_value (models/base.hpp:29; forwarded to T::Group::sample_value at models/distributions.hpp:293-298):
// draws from a group's posterior predictive, on the device, from the counter-based Philox stream.
//
// Upstream draws a parameter from the posterior and then a value from the likelihood; the marginal law of that value
// is the posterior predictive, which is what is sampled here directly:
//   bb / bbnc / dd       inverse CDF over the predictive probabilities
//   gp / bnb             inverse CDF by walking the predictive pmf upward from 0 with its ratio recurrence
//   nich                 mu' + sqrt(sigmasq' (kappa' + 1) / kappa') T,  T ~ Student-t(nu')
//   niw                  mu' + L z sqrt(dof / chi2_dof),  L L^T = psi' (kappa' + 1) / (kappa' dof), dof = nu' - d + 1
//   dm                   unsupported, as upstream ("multinomial sampling unimplemented", src/models/dm.cpp:100-111)
// Draw i of a call reads only the Philox blocks (key = seed, counter = (counter0 + i, DRAW_TAG | block)), so the result
// does not depend on how draws are spread over threads; the CPU checker restates the same sequence.
#pragma once
#include "msb_kernels.cuh"

namespace msb {

constexpr uint64_t DRAW_TAG = 0x53414d5000000000ull;  // "SAMP": keeps these counters apart from the sweeps' (row, sweep) ones
constexpr uint32_t DRAW_WALK_CAP = 1u << 26;          // longest pmf walk of the count families (bnb has no mean for a <= 1)

struct DrawStream {
  uint64_t seed, idx;
  uint32_t blk, buf[4];
  int pos;
  __device__ DrawStream(uint64_t s, uint64_t i) : seed(s), idx(i), blk(0), pos(4) {}
  __device__ uint32_t next() {
    if (pos == 4) { philox4x32_10(seed, idx, DRAW_TAG | blk, buf); blk++; pos = 0; }
    return buf[pos++];
  }
  __device__ double u53() {  // [0, 1), 53 bits
    const uint32_t a = next() >> 5, b = next() >> 6;
    return ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);
  }
  __device__ double normal() {  // Box-Muller, one of the pair
    const double u1 = u53(), u2 = u53();
    return sqrt(-2.0 * log1p(-u1)) * cos(6.283185307179586 * u2);
  }
  __device__ double gamma(double k) {  // Marsaglia-Tsang (2000), shape k, scale 1
    double boost = 1.0;
    if (k < 1.0) { boost = pow(1.0 - u53(), 1.0 / k); k += 1.0; }
    const double d = k - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    for (int it = 0; it < 1000; it++) {
      const double z = normal();
      double v = 1.0 + c * z;
      if (v <= 0.0) continue;
      v = v * v * v;
      const double u = 1.0 - u53();  // (0, 1]
      if (log(u) < 0.5 * z * z + d - d * v + d * log(v)) return boost * d * v;
    }
    return boost * d;
  }
};

// walks a pmf given p(0) and the ratio p(x + 1) / p(x) = num(x) / den(x)
template <typename RATIO>
__device__ double draw_walk(double u, double p0, RATIO ratio) {
  double t = u, p = p0;
  uint32_t x = 0;
  while (t >= p && x < DRAW_WALK_CAP) {
    t -= p;
    p *= ratio((double)x);
    x++;
    if (p == 0.0) break;
  }
  return (double)x;
}

// Posterior predictive of a niw group, set up by the whole block (mu' into mu[d], the predictive scale matrix
// psi' (kappa' + 1) / (kappa' dof) into A[d * d] and factored in place into its lower Cholesky factor L).  Returns
// dof = nu' - d + 1, or NaN when the matrix is not positive definite.  hp / ss of the group, device representation.
__device__ double niw_predictive_setup(const double *__restrict__ hp, const double *__restrict__ ss, int d, double *A,
                                       double *mu, int *s_fail, double *s_acc) {
  const double *mu0 = hp, kappa0 = hp[d], *psi0 = hp + d + 1, nu0 = hp[d + 1 + (size_t)d * d];
  const double cnt = ss[0], *sx = ss + 1, *sxx = ss + 1 + d;
  const double kn = kappa0 + cnt, nun = nu0 + cnt;
  const double dof = nun - (double)d + 1.0;
  const double scale = (kn + 1.0) / (kn * dof);
  for (int i = threadIdx.x; i < d; i += blockDim.x) mu[i] = (kappa0 * mu0[i] + sx[i]) / kn;
  __syncthreads();
  for (int e = threadIdx.x; e < d * d; e += blockDim.x) {
    const int i = e / d, j = e - i * d;
    A[e] = (psi0[e] + sxx[e] + kappa0 * mu0[i] * mu0[j] - kn * mu[i] * mu[j]) * scale;
  }
  __syncthreads();
  const double ld = block_chol_logdet(A, d, s_fail, s_acc);
  return ld != ld ? CUDART_NAN : dof;
}

// one draw of a scalar family (every family but niw and dm) from the group's posterior predictive
__device__ double draw_scalar(int family, uint32_t dim, int abi_repr, const double *__restrict__ hp,
                              const double *__restrict__ ss, DrawStream &rs) {
  if (family == FAM_BB) {
    const double p1 = (hp[0] + ss[0]) / (hp[0] + hp[1] + ss[0] + ss[1]);
    return rs.u53() < p1 ? 1.0 : 0.0;
  } else if (family == FAM_BBNC) {
    return rs.u53() < ss[0] ? 1.0 : 0.0;  // bbnc.cpp:75-83: Bernoulli(p)
  } else if (family == FAM_DD) {
    const int d = (int)dim;
    double tot = 0.0;
    for (int c = 0; c < d; c++) tot += hp[c] + ss[1 + c];
    double t = rs.u53() * tot;
    int x = d - 1;
    for (int c = 0; c < d; c++) {
      t -= hp[c] + ss[1 + c];
      if (t < 0.0) { x = c; break; }
    }
    return (double)x;
  } else if (family == FAM_GP) {  // negative binomial: a = alpha + sum, b = inv_beta + count
    const double a = hp[0] + ss[1], b = hp[1] + ss[0];
    const double p0 = exp(a * (log(b) - log1p(b)));
    const double ib = 1.0 / (1.0 + b);
    return draw_walk(rs.u53(), p0, [=](double x) { return (a + x) / (x + 1.0) * ib; });
  } else if (family == FAM_BNB) {  // beta-negative-binomial: a = alpha + r count, b = beta + sum
    const double r = hp[2], a = hp[0] + r * ss[0], b = hp[1] + ss[1];
    const double p0 = exp(lgamma(a + r) + lgamma(a + b) - lgamma(a + r + b) - lgamma(a));
    return draw_walk(rs.u53(), p0, [=](double x) { return (r + x) / (x + 1.0) * ((b + x) / (a + r + b + x)); });
  }
  // nich
  double add[3] = {ss[0], ss[1], ss[2]};
  if (abi_repr) { add[1] = ss[0] * ss[1]; add[2] = ss[2] + ss[0] * ss[1] * ss[1]; }
  const NichPost p = nich_post(hp, add);  // p.s = sqrt(lambda / nu'), lambda = kappa' / ((kappa' + 1) sigmasq')
  const double nu = hp[3] + add[0];
  const double g = rs.gamma(0.5 * nu);
  const double z = rs.normal();
  const double tv = z * sqrt(0.5 * nu / g);           // Student-t(nu')
  return p.mu + tv / (p.s * sqrt(nu));                 // scale = sqrt(1 / lambda)
}

// one niw draw mu' + L z sqrt(dof / chi2_dof) into o[d], from the factor of niw_predictive_setup (L row-major, lower
// triangle read); dof NaN gives a NaN vector
__device__ void draw_niw(DrawStream &rs, const double *__restrict__ L, const double *__restrict__ mu, double dof, int d,
                         double *__restrict__ o) {
  if (dof != dof) { for (int a = 0; a < d; a++) o[a] = CUDART_NAN; return; }
  const double g = rs.gamma(0.5 * dof);
  const double s = sqrt(0.5 * dof / g);
  for (int a = 0; a < d; a++) o[a] = mu[a];
  for (int j = 0; j < d; j++) {
    const double z = rs.normal() * s;
    for (int a = j; a < d; a++) o[a] += L[a * d + j] * z;
  }
}

// ss in the device representation (nich: [n, sum x, sum x^2]); `abi_repr` != 0: nich arrives as (count, mean,
// count_times_variance) like msb_value_* hands it over.  out[i * width + j], width = dim (niw) or 1.
__global__ void sample_value_kernel(int family, uint32_t dim, int abi_repr, const double *__restrict__ hp,
                                    const double *__restrict__ ss, uint64_t seed, uint64_t counter0, size_t n,
                                    double *__restrict__ out) {
  extern __shared__ double sm[];
  __shared__ int s_fail;
  __shared__ double s_acc;
  const int d = (int)dim;
  double dof = 0.0;
  if (family == FAM_NIW) dof = niw_predictive_setup(hp, ss, d, sm, sm + d * d, &s_fail, &s_acc);  // the whole block, once
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    DrawStream rs(seed, counter0 + i);
    if (family == FAM_NIW) draw_niw(rs, sm, sm + d * d, dof, d, out + i * (size_t)d);
    else out[i] = draw_scalar(family, dim, abi_repr, hp, ss, rs);
  }
}

// niw predictive factors of every group for the batched imputation (impute_kernel): one block per group column k;
// fac + slot * (d * d + d + 1) = [L (d x d, lower triangle) | mu' (d) | dof], the same setup as sample_value_kernel's,
// so that a cell's draw is mu' + L z sqrt(dof / chi2) without a factorisation per cell
__global__ void niw_predictive_factor_kernel(FeatDev f, const double *__restrict__ hp, const double *__restrict__ ss,
                                             const int32_t *__restrict__ col2slot, double *__restrict__ fac) {
  extern __shared__ double sm[];
  __shared__ int s_fail;
  __shared__ double s_acc;
  const int d = (int)f.dim;
  const int slot = col2slot[blockIdx.x];
  const double dof = niw_predictive_setup(hp + f.hp_off, ss + f.ss_off + (size_t)slot * f.ss_w, d, sm, sm + d * d, &s_fail, &s_acc);
  double *o = fac + (size_t)slot * ((size_t)d * d + d + 1);
  for (int e = threadIdx.x; e < d * d + d; e += blockDim.x) o[e] = sm[e];
  if (threadIdx.x == 0) o[d * d + d] = dof;
}

// Batched posterior-predictive imputation, one thread per (row, feature): an observed cell is copied from the value
// column (the cast value the device holds), a masked one -- masked as the scorer sees it: dd categories outside
// [0, C), a niw vector with any masked element -- is drawn from the predictive of the group the sampler put in
// new_slot[i], from the Philox stream (seed, cbase + (id0 + i) D + d): the draw msb_state_sample_value makes with that
// counter and n = 1.  A masked dm cell sets *unsupported (dm.cpp:100-111 has no sampler).
struct ImputeFeat { uint64_t off; const double *fac; };  // first output column; niw: the factors of niw_predictive_factor_kernel
__global__ void impute_kernel(const FeatDev *__restrict__ feats, const ImputeFeat *__restrict__ ifeat, int nfeat,
                              const double *__restrict__ hp, const double *__restrict__ ss, const int32_t *__restrict__ new_slot,
                              size_t row_lo, size_t nrows, uint64_t seed, uint64_t cbase, uint64_t id0, double *__restrict__ out,
                              size_t ld, uint32_t *__restrict__ unsupported) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int d = blockIdx.y;
  if (i >= nrows) return;
  const FeatDev &f = feats[d];
  const size_t row = row_lo + i;
  double *o = out + i * ld + ifeat[d].off;
  bool masked;
  if (f.kind == KIND_TABLE) {
    uint32_t x;
    if (f.coltype == COL_U8) x = ((const uint8_t *)f.col)[row];
    else if (f.coltype == COL_U16) x = ((const uint16_t *)f.col)[row];
    else x = ((const uint32_t *)f.col)[row];
    masked = x >= f.ncat;
    if (!masked) o[0] = (double)x;
  } else if (f.kind == KIND_GP) {
    const uint32_t x = ((const uint32_t *)f.col)[row];
    masked = x == GP_SENTINEL;
    if (!masked) o[0] = (double)x;
  } else if (f.kind == KIND_NICH) {
    const float x = ((const float *)f.col)[row];
    masked = x != x;
    if (!masked) o[0] = (double)x;
  } else if (f.kind == KIND_NIW) {
    const float *x = (const float *)f.col + row * (size_t)f.dim;
    masked = x[0] != x[0];
    if (!masked) for (uint32_t a = 0; a < f.dim; a++) o[a] = (double)x[a];
  } else {  // dm: a row of counts, sentinel in element 0 when masked
    const uint32_t *x = (const uint32_t *)f.col + row * (size_t)f.dim;
    masked = x[0] == GP_SENTINEL;
    if (masked) { atomicOr(unsupported, 1u); for (uint32_t a = 0; a < f.dim; a++) o[a] = CUDART_NAN; return; }
    for (uint32_t a = 0; a < f.dim; a++) o[a] = (double)x[a];
  }
  if (!masked) return;
  const int slot = new_slot[i];
  DrawStream rs(seed, cbase + (id0 + i) * (uint64_t)nfeat + (uint64_t)d);
  if (f.kind == KIND_NIW) {
    const int dd = (int)f.dim;
    const double *fac = ifeat[d].fac + (size_t)slot * ((size_t)dd * dd + dd + 1);
    draw_niw(rs, fac, fac + dd * dd, fac[dd * dd + dd], dd, o);
  } else {
    o[0] = draw_scalar(f.family, f.dim, 0, hp + f.hp_off, ss + f.ss_off + (size_t)slot * f.ss_w, rs);
  }
}

}  // namespace msb
