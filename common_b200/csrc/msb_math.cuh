// msb_math.cuh -- device math shared by the kernels of the hot path.
//
// Closed forms of the conjugate families the reference reaches through
// distributions_group<T>::score_value (include/microscopes/models/
// distributions.hpp:280-285 in the reference tree); the maths itself lives in
// the un-vendored `distributions` library and is restated from the published
// posterior-predictive formulas (SURVEY.md section 8a).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <math_constants.h>

namespace msb {

enum Family : int { FAM_BB = 0, FAM_BNB = 1, FAM_GP = 2, FAM_NICH = 3, FAM_DD = 4, FAM_NIW = 5, FAM_BBNC = 6, FAM_DM = 7 };

// ---------------------------------------------------------------------------
// msb_expf: exp() built only from correctly rounded IEEE-754 binary32
// operations in a fixed order, so that the CPU checker can reproduce it bit for
// bit (sampler contract, DESIGN.md).  Explicit _rn intrinsics are never
// contracted or reassociated by nvcc.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float msb_expf(float x) {
  // branch-free: the polynomial runs on the clamped argument and the out-of-range result is selected at the end
  const float x_in = x;
  x = fminf(fmaxf(x, -104.0f), 88.0f);
  // rint and the float -> int conversion by the 1.5 * 2^23 trick (two FADDs on the FMA pipe instead of FRND + F2I
  // on the quarter-rate XU pipe); identical to rintf / (int) for |x log2e| < 2^22, and x is in [-104, 88] here
  const float kbias = __fadd_rn(__fmul_rn(x, 1.44269504f), 12582912.0f);
  const float kf = __fsub_rn(kbias, 12582912.0f);
  float r = __fmaf_rn(kf, -0.693145752f, x);
  r = __fmaf_rn(kf, -1.42860677e-6f, r);
  float p = 1.9875691500e-4f;
  p = __fmaf_rn(p, r, 1.3981999507e-3f);
  p = __fmaf_rn(p, r, 8.3334519073e-3f);
  p = __fmaf_rn(p, r, 4.1665795894e-2f);
  p = __fmaf_rn(p, r, 1.6666665459e-1f);
  p = __fmaf_rn(p, r, 5.0000001201e-1f);
  const float r2 = __fmul_rn(r, r);
  p = __fmaf_rn(p, r2, r);
  p = __fadd_rn(p, 1.0f);
  const int k = __float_as_int(kbias) - 0x4B400000;
  // p * 2^k with a single rounding: p is in (0.5, 2), so for kk = max(k, -125) the product p * 2^kk is a normal
  // number and adding kk to the exponent field is exact; the remaining factor 2^(k - kk) (!= 1 only for results in
  // the subnormal range) is one correctly rounded multiply.  Same bits as the checker's (p * 2^(k/2)) * 2^(k - k/2):
  // both are exact up to that one final rounding.
  const int kk = max(k, -125);
  const float pk = __int_as_float(__float_as_int(p) + (kk << 23));
  const float y = __fmul_rn(pk, __int_as_float((k - kk + 127) << 23));
  return x_in >= -104.0f ? y : (x_in != x_in ? x_in : 0.0f);
}

// msb_expf of two arguments that both lie in [-86, 0] (not NaN), with the packed fp32 instructions of sm_100
// (FMUL2 / FADD2 / FFMA2: one issue slot per pair).  The same operations in the same order, so the same bits:
//   * the clamp and the final select are identities on that range, and a - b is a + (-b) in IEEE arithmetic;
//   * k = rint(x log2e) is in [-124, 0], so kk = max(k, -125) = k and the subnormal factor 2^(k - kk) is 1;
//   * kbias = 1.5 * 2^23 + k has the bits 0x4B400000 + k, and 0x4B400000 << 23 is 0 mod 2^32, so adding
//     kbias_bits << 23 to p's bits adds exactly k << 23 to its exponent field.
// The one exception is the add of 1.5 * 2^23 to x log2e, kept as two scalar FADDs: ptxas contracts mul.rn.f32x2
// followed by add.rn.f32x2 into one FFMA2 despite the rounding modifiers, and the fused form can round k differently.
// Checked over every float of the range against msb_expf by msb_selftest_expf2.
__device__ __forceinline__ float2 msb_expf2_dense(float2 x) {
  const float2 xl = __fmul2_rn(x, make_float2(1.44269504f, 1.44269504f));
  const float2 kbias = make_float2(__fadd_rn(xl.x, 12582912.0f), __fadd_rn(xl.y, 12582912.0f));
  const float2 kf = __fadd2_rn(kbias, make_float2(-12582912.0f, -12582912.0f));
  float2 r = __ffma2_rn(kf, make_float2(-0.693145752f, -0.693145752f), x);
  r = __ffma2_rn(kf, make_float2(-1.42860677e-6f, -1.42860677e-6f), r);
  float2 p = __ffma2_rn(make_float2(1.9875691500e-4f, 1.9875691500e-4f), r, make_float2(1.3981999507e-3f, 1.3981999507e-3f));
  p = __ffma2_rn(p, r, make_float2(8.3334519073e-3f, 8.3334519073e-3f));
  p = __ffma2_rn(p, r, make_float2(4.1665795894e-2f, 4.1665795894e-2f));
  p = __ffma2_rn(p, r, make_float2(1.6666665459e-1f, 1.6666665459e-1f));
  p = __ffma2_rn(p, r, make_float2(5.0000001201e-1f, 5.0000001201e-1f));
  const float2 r2 = __fmul2_rn(r, r);
  p = __ffma2_rn(p, r2, r);
  p = __fadd2_rn(p, make_float2(1.0f, 1.0f));
  return make_float2(__int_as_float(__float_as_int(p.x) + (__float_as_int(kbias.x) << 23)),
                     __int_as_float(__float_as_int(p.y) + (__float_as_int(kbias.y) << 23)));
}

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11).  key = seed, counter = (row, sweep).
// ---------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox4x32_10(uint64_t seed, uint64_t row, uint64_t sweep, uint32_t out[4]) {
  uint32_t c0 = (uint32_t)row, c1 = (uint32_t)(row >> 32), c2 = (uint32_t)sweep, c3 = (uint32_t)(sweep >> 32);
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__host__ __device__ __forceinline__ float philox_u01(uint64_t seed, uint64_t row, uint64_t sweep) {
  uint32_t r[4];
  philox4x32_10(seed, row, sweep, r);
  return (float)(r[0] >> 8) * 5.9604644775390625e-8f;  // [0,1)
}

// ---------------------------------------------------------------------------
// fp64 closed forms over the device suffstat representation (all additive):
//   bb   ss = [heads, tails]                 hp = [alpha, beta]
//   dd   ss = [count_sum, counts[dim]]       hp = alphas[dim]   (asum passed in)
//   gp   ss = [count, sum, log_prod]         hp = [alpha, inv_beta]
//   bnb  ss = [count, sum]                   hp = [alpha, beta, r]
//   nich ss = [count, sum x, sum x^2]        hp = [mu, kappa, sigmasq, nu]
// ---------------------------------------------------------------------------
__device__ __forceinline__ double bb_score(const double *hp, const double *ss, int x) {
  const double a = hp[0] + ss[0], b = hp[1] + ss[1];
  return log((x ? a : b) / (a + b));
}
// bbnc (src/models/bbnc.cpp:46-53): the group holds its own success probability p; ss = [p, heads, tails]
__device__ __forceinline__ double bbnc_score(const double *ss, int x) { return x ? log(ss[0]) : log1p(-ss[0]); }
__device__ __forceinline__ double dd_score(const double *hp, double asum, const double *ss, uint32_t x) {
  return log((hp[x] + ss[1 + x]) / (asum + ss[0]));
}
struct GpPost { double a, b, ca, l1pb; };  // ca = -lgamma(a) + a log b - a log1p(b)
__device__ __forceinline__ GpPost gp_post(const double *hp, const double *ss) {
  GpPost p;
  p.a = hp[0] + ss[1];
  p.b = hp[1] + ss[0];
  p.l1pb = log1p(p.b);
  p.ca = -lgamma(p.a) + p.a * log(p.b) - p.a * p.l1pb;
  return p;
}
__device__ __forceinline__ double gp_score(const GpPost &p, double x) {
  return lgamma(p.a + x) - lgamma(x + 1.0) + p.ca - x * p.l1pb;
}
// bnb (beta-negative-binomial): hp = [alpha, beta, r], ss = [count, sum]; posterior Beta(a, b) over the success
// probability with a = alpha + r count, b = beta + sum; predictive
//   lgamma(r + x) - lgamma(r) - lgamma(x + 1) + lbeta(a + r, b + x) - lbeta(a, b)
struct BnbPost { double ar, b, r, c; };  // ar = a + r, c = -lgamma(r) - lbeta(a, b) + lgamma(a + r)
__device__ __forceinline__ BnbPost bnb_post(const double *hp, const double *ss) {
  BnbPost p;
  const double a = hp[0] + hp[2] * ss[0];
  p.b = hp[1] + ss[1];
  p.r = hp[2];
  p.ar = a + p.r;
  p.c = -lgamma(p.r) - (lgamma(a) + lgamma(p.b) - lgamma(a + p.b)) + lgamma(p.ar);
  return p;
}
__device__ __forceinline__ double bnb_score(const BnbPost &p, double x) {
  return lgamma(p.r + x) - lgamma(x + 1.0) + lgamma(p.b + x) - lgamma(p.ar + p.b + x) + p.c;
}
struct NichPost { double mu, s, c1, c0; };  // score = c0 + c1 * log1p(((x - mu) s)^2)
__device__ __forceinline__ NichPost nich_post(const double *hp, const double *ss) {
  const double n = ss[0];
  const double mean = n > 0.0 ? ss[1] / n : 0.0;
  double ctv = n > 0.0 ? ss[2] - ss[1] * mean : 0.0;
  if (ctv < 0.0) ctv = 0.0;
  const double mu1 = hp[0] - mean;
  const double kappa = hp[1] + n;
  const double nu = hp[3] + n;
  const double sigmasq = (hp[3] * hp[2] + ctv + (n * hp[1] * mu1 * mu1) / kappa) / nu;
  const double lambda = kappa / ((kappa + 1.0) * sigmasq);
  NichPost p;
  p.mu = (hp[1] * hp[0] + mean * n) / kappa;
  p.s = sqrt(lambda / nu);
  p.c1 = -0.5 * nu - 0.5;
  p.c0 = lgamma(0.5 * nu + 0.5) - lgamma(0.5 * nu) + 0.5 * log(lambda / (CUDART_PI * nu));
  return p;
}
__device__ __forceinline__ double nich_score(const NichPost &p, double x) {
  const double t = (x - p.mu) * p.s;
  return p.c0 + p.c1 * log1p(t * t);
}

// dm (src/models/dm.cpp:38-76): lgamma(e + x) - lgamma(e) for a count x; the product form for small x has no
// cancellation (e can be in the thousands)
__device__ __forceinline__ double lgamma_rise(double e, uint32_t x) {
  if (x <= 12u) {
    double p = 1.0;
    for (uint32_t j = 0; j < x; j++) p *= e + (double)j;
    return log(p);
  }
  return lgamma(e + (double)x) - lgamma(e);
}

// fp32 log2(1 + z), z >= 0, for the nich inner loop (the natural-log factor ln 2 is folded into the
// per-(group, feature) coefficient c1 by build_params_kernel).  z < 1/16: z times a degree-3 polynomial on the
// FMA pipe -- the interpolant of log2(1 + z) / z at the Chebyshev nodes of [0, 1/16]: approximation error 2.4e-8,
// 1.3e-7 relative once evaluated in fp32 (the degree-5 Taylor form it replaces: 1.15e-7, two more FFMA per unit);
// above: MUFU.LG2(1 + z), whose absolute error 2^-22 is at most 2.7e-6 relative just above the switch.
// Branch-free: both are evaluated and selected.
// MUFU.LG2 without the subnormal-input fix-up __log2f carries (the argument here is 1 + z >= 1)
__device__ __forceinline__ float lg2_ftz(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
#define MSB_L1P_C0 1.442695022e+00f
#define MSB_L1P_C1 -7.213315964e-01f
#define MSB_L1P_C2 4.796128273e-01f
#define MSB_L1P_C3 -3.270350397e-01f
__device__ __forceinline__ float log2_1p_pos(float z) {
  float p = MSB_L1P_C3;
  p = fmaf(p, z, MSB_L1P_C2);
  p = fmaf(p, z, MSB_L1P_C1);
  p = fmaf(p, z, MSB_L1P_C0);
  const float small = p * z;
  const float big = lg2_ftz(1.0f + z);
  return z < 0.0625f ? small : big;
}

// The same for two groups at once with the packed fp32 instructions of sm_100 (FADD2 / FMUL2 / FFMA2: one issue
// slot per pair): the nich loop is bound by instruction issue, not by the FMA lanes.  Bit-identical to two
// calls of log2_1p_pos.
__device__ __forceinline__ float2 log2_1p_pos2(float2 z) {
  float2 p = __ffma2_rn(make_float2(MSB_L1P_C3, MSB_L1P_C3), z, make_float2(MSB_L1P_C2, MSB_L1P_C2));
  p = __ffma2_rn(p, z, make_float2(MSB_L1P_C1, MSB_L1P_C1));
  p = __ffma2_rn(p, z, make_float2(MSB_L1P_C0, MSB_L1P_C0));
  const float2 small = __fmul2_rn(p, z);
  const float2 w = __fadd2_rn(z, make_float2(1.0f, 1.0f));
  return make_float2(z.x < 0.0625f ? small.x : lg2_ftz(w.x), z.y < 0.0625f ? small.y : lg2_ftz(w.y));
}

}  // namespace msb
