// simplyp_bands.cuh — arithmetic of the posterior predictive bands (simplyp_predictive_draws_device,
// simplyp_nanquantile_device, include/simplyp_b200.h).
//
// sim_series_value: the simulated counterpart of an observed series kind, shared by the calibration kernel's fused
// statistics (CalIO::emit) and the draw kernel, so the bands see exactly the values the statistics and the sampler
// see.
//
// band_epsilon: the standard normal deviate of the likelihood's error model N(o; s, (m s)^2) for one (member, day,
// series), by Box-Muller from one Philox4x32-10 block keyed by the seed with counter (member, day, series, 2).  The
// sampler (simplyp_mcmc.cuh) only uses blocks 0 and 1 of that word, so the two streams never share a counter.
//
// The index and interpolation arithmetic of np.nanquantile(x, q, method='linear') (NumPy 2.3, _quantile / _lerp):
// v = (n - 1) q, i = floor(v), g = v - i; when v >= n - 1 both neighbours are the last value and NumPy's index is -1,
// so g = v - (-1); then b - (b - a)(1 - g) if g >= 0.5 else a + (b - a) g, every operation rounded on its own
// (an infinite neighbour therefore gives NaN, as in NumPy).
//
// Inline __host__ __device__ code like simplyp_mcmc.cuh: the CPU test tier compiles it for the host.
#pragma once

#include <cstring>

#include "simplyp_mcmc.cuh"

namespace simplyp {

// Q_cumecs = Qr*A*1000/86400 and the concentrations (flux/Qr)/A_catch in the reference's order of operations
// (model.py:784-793, :840-845); rQ = sp_rcp(Qr), rA = sp_rcp(A).  The quotients are formed by sp_div: see the
// comment in CalIO::emit (simplyp_kernels.cu) for why.
SP_HD double sim_series_value(int kind, double Qr, double msus, double tdp, double pp, double A, double rQ, double rA,
                              double f_TDP) {
  switch (kind) {
    case SIMPLYP_V_Q:   return sp_div(Qr * A * 1000.0, 86400.0, 1.0 / 86400.0);
    case SIMPLYP_V_SS:  return sp_div(sp_div(msus, Qr, rQ), A, rA);
    case SIMPLYP_V_TDP: return sp_div(sp_div(tdp, Qr, rQ), A, rA);
    case SIMPLYP_V_PP:  return sp_div(sp_div(pp, Qr, rQ), A, rA);
    case SIMPLYP_V_TP:  return sp_div(sp_div(tdp, Qr, rQ), A, rA) + sp_div(sp_div(pp, Qr, rQ), A, rA);
    default:            return sp_div(sp_div(tdp, Qr, rQ), A, rA) * f_TDP;
  }
}

constexpr uint32_t BAND_BLOCK = 2;   // the fourth counter word of the error draws (the sampler uses 0 and 1)

SP_HD void band_words(uint64_t seed, int member, int day, int series, uint32_t (&r)[4]) {
  const uint32_t ctr[4] = {(uint32_t)member, (uint32_t)day, (uint32_t)series, BAND_BLOCK};
  philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32), r);
}

// cos(pi x) for 0 <= x < 2.  The device has cospi; glibc has none, so the host reduces x to r = x - n/2 with
// |r| <= 1/4 (exact) and takes cos or sin of pi r, which keeps the result within a few ulp everywhere.
SP_HD double band_cospi(double x) {
#if defined(__CUDA_ARCH__)
  return cospi(x);
#else
  const double n = nearbyint(2.0 * x);
  const double t = M_PI * (x - 0.5 * n);
  switch ((int)n & 3) {
    case 0:  return cos(t);
    case 1:  return -sin(t);
    case 2:  return -cos(t);
    default: return sin(t);
  }
#endif
}

// Box-Muller: u1 = 1 - u53(r0, r1) in (0, 1], u2 = u53(r2, r3), eps = sqrt(-2 ln u1) cos(2 pi u2).
SP_HD double band_epsilon(uint64_t seed, int member, int day, int series) {
  uint32_t r[4];
  band_words(seed, member, day, series, r);
  const double u1 = 1.0 - mcmc_u53(r[0], r[1]);
  const double u2 = mcmc_u53(r[2], r[3]);
  return sqrt(-2.0 * log(u1)) * band_cospi(2.0 * u2);
}

// y = sim + (m sim) eps, without FMA contraction.
SP_HD double band_draw(double sim, double m, double eps) { return mc_add(sim, mc_mul(mc_mul(m, sim), eps)); }

// ---- np.nanquantile (method 'linear')
// Order-preserving 64-bit key of a double: -inf < ... < -0 < +0 < ... < +inf < every NaN.
SP_HD uint64_t nq_bits(double x) {
#if defined(__CUDA_ARCH__)
  return (uint64_t)__double_as_longlong(x);
#else
  uint64_t b;
  memcpy(&b, &x, sizeof b);
  return b;
#endif
}
SP_HD uint64_t nq_key(double x) {
  if (x != x) return ~0ull;
  const uint64_t b = nq_bits(x);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
SP_HD double nq_value(uint64_t k) {
  const uint64_t b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)b);
#else
  double x;
  memcpy(&x, &b, sizeof x);
  return x;
#endif
}

// Positions of the two neighbours (0-based, in the sorted non-NaN values) and the weight g for quantile q of n >= 1
// values.
SP_HD void nq_index(long long n, double q, long long* lo, long long* hi, double* g) {
  const double v = mc_mul((double)(n - 1), q);
  if (v >= (double)(n - 1)) {
    *lo = *hi = n - 1;
    *g = mc_sub(v, -1.0);
  } else {
    const double f = floor(v);
    *lo = (long long)f;
    *hi = *lo + 1;
    *g = mc_sub(v, f);
  }
}

// NumPy's _lerp(a, b, g).
SP_HD double nq_lerp(double a, double b, double g) {
  const double d = mc_sub(b, a);
  return (g >= 0.5) ? mc_sub(b, mc_mul(d, mc_sub(1.0, g))) : mc_add(a, mc_mul(d, g));
}

}  // namespace simplyp
