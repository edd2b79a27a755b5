// simplyp_mcmc.cuh — per-walker arithmetic of the ensemble sampler (simplyp_mcmc_*_device, include/simplyp_b200.h).
//
// The affine-invariant stretch move of Goodman & Weare (2010) as emcee's default StretchMove runs it: the walkers are
// split into the contiguous halves [0, W/2) and [W/2, W); each walker of the active half draws a partner j from the
// other half and a stretch factor z with density ~ 1/sqrt(z) on [1/a, a], proposes y = x_j - z (x_j - x_k) and accepts
// with probability min(1, z^(K-1) p(y) / p(x_k)).  The random words come from Philox4x32-10 (Salmon et al. 2011, the
// generator and constants of cuRAND's curand_Philox4x32_10) keyed by the seed, with counter
// (walker, iteration lo, iteration hi, block): every draw is a pure function of (seed, walker, iteration), so a run
// does not depend on launch geometry and a continued run draws what a longer one would have drawn.
//
// Inline __host__ __device__ code like simplyp_core.cuh: the test harness (tests/hostemu) compiles it for the host.
// z and y are formed with explicitly rounded operations so that nvcc cannot contract them into FMAs and a NumPy
// restatement reproduces the proposals bit for bit.
#pragma once

#include "simplyp_core.cuh"

namespace simplyp {

SP_HD double mc_add(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
SP_HD double mc_sub(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dsub_rn(a, b);
#else
  return a - b;
#endif
}
SP_HD double mc_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
SP_HD double mc_div(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __ddiv_rn(a, b);
#else
  return a / b;
#endif
}
SP_HD uint32_t mc_mulhi(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

// Philox4x32-10: ten rounds, the key bumped between rounds (cuRAND's curand_Philox4x32_10(uint4, uint2)).
SP_HD void philox4x32_10(const uint32_t (&ctr)[4], uint32_t k0, uint32_t k1, uint32_t (&out)[4]) {
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
  for (int r = 0; r < 10; ++r) {
    if (r > 0) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    const uint32_t hi0 = mc_mulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = mc_mulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// The four words of block b (0: partner and stretch, 1: acceptance) of walker w at iteration t.
SP_HD void mcmc_words(uint64_t seed, long long t, int w, int b, uint32_t (&r)[4]) {
  const uint64_t ut = (uint64_t)t;
  const uint32_t ctr[4] = {(uint32_t)w, (uint32_t)ut, (uint32_t)(ut >> 32), (uint32_t)b};
  philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32), r);
}

// A uniform double in [0, 1) on the 2^-53 grid from 27 + 26 bits of two words (exact in any rounding mode).
SP_HD double mcmc_u53(uint32_t a, uint32_t b) {
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// z = ((a - 1) u + 1)^2 / a
SP_HD double mcmc_stretch_z(double u, double a) {
  const double s = mc_add(mc_mul(mc_sub(a, 1.0), u), 1.0);
  return mc_div(mc_mul(s, s), a);
}

// Proposal of walker k of the active half (rows [half*H, half*H + H) of walkers [W][K]) at iteration t: writes prop[K]
// and ln z, and returns 1 if the proposal lies outside the prior box [lo, hi] (or is not a number).
SP_HD int mcmc_propose_walker(const SimplypMcmc& mc, const double* walkers, long long t, int half, int k,
                              double* prop, double* log_z) {
  const int W = mc.n_walkers, H = W / 2, K = mc.n_free;
  const int w = half * H + k;
  uint32_t r[4];
  mcmc_words(mc.seed, t, w, 0, r);
  const int j = (1 - half) * H + (int)(((uint64_t)r[0] * (uint64_t)H) >> 32);
  const double z = mcmc_stretch_z(mcmc_u53(r[1], r[2]), mc.stretch);
  *log_z = log(z);
  const double* xk = walkers + (size_t)w * K;
  const double* xj = walkers + (size_t)j * K;
  int out = 0;
  for (int i = 0; i < K; ++i) {
    const double y = mc_sub(xj[i], mc_mul(z, mc_sub(xj[i], xk[i])));
    prop[i] = y;
    if (!(y >= mc.param[i].lo && y <= mc.param[i].hi)) out = 1;
  }
  return out;
}

// Writes value v of free parameter p into the member's parameter row mrow[NP_MEMBER] or its sub-catchment rows
// srow[S][NP_SC] (the sampler's proposals, the DE trials and the Sobol' design all place their values this way).  An
// error-model parameter (SIMPLYP_MCMC_ERROR_MODEL) is in no row: simplyp_calibrate_ar1_device reads it where it is.
SP_HD void mcmc_write_target(const SimplypMcmcParam& p, int S, double v, double* mrow, double* srow) {
  if (p.kind == SIMPLYP_MCMC_MEMBER) {
    mrow[p.index] = v;
  } else if (p.kind == SIMPLYP_MCMC_SC_AT) {
    srow[(size_t)p.pos * SIMPLYP_NP_SC + p.index] = v;
  } else if (p.kind == SIMPLYP_MCMC_SC_ALL) {
    for (int s = 0; s < S; ++s) srow[(size_t)s * SIMPLYP_NP_SC + p.index] = v;
  }
}

// Log-probability of one member from its fused statistics: the sum of the Gaussian log-likelihoods of its V series
// (stats row [V][SIMPLYP_NSTAT]), or -inf if the integration of any of its S sub-catchments raised a status bit
// (diag row [S][SIMPLYP_NDIAG]) or the sum is not a number.  The uniform prior adds 0 inside the box.
SP_HD double mcmc_member_lp(const double* stats, int V, const int64_t* diag, int S) {
  for (int s = 0; s < S; ++s)
    if (diag[(size_t)s * SIMPLYP_NDIAG + SIMPLYP_DG_STATUS] != 0) return -INFINITY;
  double lp = 0.0;
  for (int v = 0; v < V; ++v) lp = mc_add(lp, stats[(size_t)v * SIMPLYP_NSTAT + SIMPLYP_ST_LOGLIK]);
  return lp == lp ? lp : -INFINITY;
}

// Metropolis-Hastings step of walker k of the active half: accepts prop[K] (log-probability lp_new) if
// ln u' < (K - 1) ln z + lp_new - lp[w]; updates walkers, lp and accepted.  Returns 1 on acceptance.
SP_HD int mcmc_accept_walker(const SimplypMcmc& mc, long long t, int half, int k, double lp_new, double log_z,
                             const double* prop, double* walkers, double* lp, int64_t* accepted) {
  const int H = mc.n_walkers / 2, K = mc.n_free;
  const int w = half * H + k;
  uint32_t r[4];
  mcmc_words(mc.seed, t, w, 1, r);
  const double log_u = log(mcmc_u53(r[0], r[1]));
  const double diff = mc_sub(mc_add(mc_mul((double)(K - 1), log_z), lp_new), lp[w]);
  if (!(log_u < diff)) return 0;
  for (int i = 0; i < K; ++i) walkers[(size_t)w * K + i] = prop[i];
  lp[w] = lp_new;
  accepted[w] += 1;
  return 1;
}

}  // namespace simplyp
