// simplyp_ar1.cuh — the autocorrelated (AR(1)) error model of the log-likelihood (simplyp_calibrate_ar1_device,
// include/simplyp_b200.h).
//
// For a series with observed days t_1 < ... < t_n (observation o_i, simulated value s_i, error scale m of its kind):
//   eta_i = (o_i - s_i) / sigma_i,  sigma_i = m s_i   (the standardised residual of the iid likelihood)
//   rho_1 = 0,  rho_i = phi^(t_i - t_{i-1})
//   l = sum_i [ -1/2 ln 2pi - ln sigma_i - 1/2 ln(1 - rho_i^2) - (eta_i - rho_i eta_{i-1})^2 / (2 (1 - rho_i^2)) ]
// which is the exact log-density of N(s, Sigma) with Sigma_ij = sigma_i sigma_j phi^|t_i - t_j| (Schoups & Vrugt 2010,
// the Gaussian member of their generalised likelihood): a stationary AR(1) sampled at irregular days is Markov, so the
// sparse chemistry series need no gap filling.  phi = 0 gives the iid value.  A series with no observed day gives 0;
// |phi| >= 1 (or NaN), s <= 0, sigma <= 0 or a non-finite sum give -inf, as the iid likelihood's NaN -> -inf rule does.
//
// The per-term arithmetic is inline __host__ __device__ code like simplyp_bands.cuh, every operation rounded on its own
// (mc_*), so the CPU test tier's host build differs from the device only in the last bits of log.  The kernel (one warp
// per (member, series) row) is compiled by nvcc only.
#pragma once

#include "simplyp_mcmc.cuh"

namespace simplyp {

constexpr int AR1_WARPS = 8;   // rows per block of ar1_loglik_kernel

// phi^gap for gap >= 1 by repeated squaring: the same multiplications on the host and on the device.
SP_HD double ar1_rho(double phi, int gap) {
  double r = 1.0, b = phi;
  for (unsigned g = (unsigned)gap; g != 0u; g >>= 1) {
    if (g & 1u) r = mc_mul(r, b);
    b = mc_mul(b, b);
  }
  return r;
}

// The standardised residual eta of one observed day; *sigma receives m s.
SP_HD double ar1_eta(double o, double s, double m, double* sigma) {
  const double sg = mc_mul(m, s);
  *sigma = sg;
  return mc_div(mc_sub(o, s), sg);
}

// The term of one observed day from its eta and sigma, the predecessor's eta and rho (rho = 0, eta_prev = 0 for the
// first observed day).  NaN where the density is undefined: s <= 0, sigma <= 0, or anything not a number.
SP_HD double ar1_term(double s, double sigma, double eta, double rho, double eta_prev) {
  if (!(s > 0.0) || !(sigma > 0.0)) return NAN;
  const double q = mc_mul(mc_sub(1.0, rho), mc_add(1.0, rho));           // 1 - rho^2, exact digits near |rho| = 1
  const double u = mc_sub(eta, mc_mul(rho, eta_prev));
  const double t = mc_sub(mc_sub(-0.91893853320467274178, log(sigma)), mc_mul(0.5, log(q)));
  return mc_sub(t, mc_div(mc_mul(u, u), mc_mul(2.0, q)));
}

SP_HD bool ar1_phi_valid(double phi) { return fabs(phi) < 1.0; }   // false for NaN

// The row's value from its sum over the observed days.
SP_HD double ar1_finish(double phi, double sum) {
  if (!ar1_phi_valid(phi)) return -INFINITY;
  return (sum - sum == 0.0) ? sum : -INFINITY;                        // NaN or +-inf -> -inf
}

#if defined(__CUDACC__)
// One warp per row (member m, series v) of stats[M][V][SIMPLYP_NSTAT] whose ar.col[v] >= 0: overwrites its LOGLIK.
// The days are walked in chunks of 32, day d on lane d % 32: a ballot of the observed lanes gives each lane its
// predecessor in the chunk (its eta by a shuffle); the chunk's last observed (day, eta) carries to the next chunk.
// Each lane sums its own terms in day order, then a fixed xor tree adds the 32 partial sums: the value depends on
// neither M nor the member order nor the launch.
__global__ void __launch_bounds__(AR1_WARPS * 32) ar1_loglik_kernel(const double* sim_obs, const double* obs,
                                                                    const int32_t* obs_desc, const double* member_params,
                                                                    const SimplypAr1 ar, long long M, int V, int D,
                                                                    double* stats) {
  const long long row = (long long)blockIdx.x * AR1_WARPS + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M * V) return;
  const long long m = row / V;
  const int v = (int)(row - m * V);
  const int c = ar.col[v];
  if (c < 0) return;
  const double phi = ar.phi[m * ar.row_stride + c];
  const int kind = obs_desc[2 * v + 1];
  const double em = member_params[m * SIMPLYP_NP_MEMBER + SIMPLYP_P_ERR_M0 + kind];
  const double* o_row = obs + (size_t)v * D;
  const double* s_row = sim_obs + (size_t)row * D;
  const unsigned FULL = 0xffffffffu;
  double acc = 0.0, last_eta = 0.0;
  int last_day = -1;
  if (ar1_phi_valid(phi)) {
    for (int d0 = 0; d0 < D; d0 += 32) {
      const int d = d0 + lane;
      const double o = d < D ? __ldg(o_row + d) : NAN;
      const bool seen = o == o;
      const unsigned mask = __ballot_sync(FULL, seen);
      if (mask == 0u) continue;
      const double s = seen ? __ldcs(s_row + d) : 1.0;
      double sg;
      const double eta = ar1_eta(seen ? o : 1.0, s, em, &sg);
      const unsigned below = mask & ((1u << lane) - 1u);
      const int pl = below ? 31 - __clz(below) : lane;
      const double eta_pl = __shfl_sync(FULL, eta, pl);
      if (seen) {
        const int pred = below ? d0 + pl : last_day;
        const double rho = pred < 0 ? 0.0 : ar1_rho(phi, d - pred);
        const double eta_prev = below ? eta_pl : (pred < 0 ? 0.0 : last_eta);
        acc = mc_add(acc, ar1_term(s, sg, eta, rho, eta_prev));
      }
      const int hi = 31 - __clz(mask);
      last_eta = __shfl_sync(FULL, eta, hi);
      last_day = d0 + hi;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc = mc_add(acc, __shfl_xor_sync(FULL, acc, off));
  if (lane == 0) stats[(size_t)row * SIMPLYP_NSTAT + SIMPLYP_ST_LOGLIK] = ar1_finish(phi, acc);
}
#endif

}  // namespace simplyp
