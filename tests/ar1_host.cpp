// TEST HARNESS ONLY — compiles simplyp_ar1.cuh (the AR(1) error model's per-term arithmetic) and the sampler's
// parameter-row writes (simplyp_mcmc.cuh) for the host, so that the CPU-only test tier can check them against NumPy
// without a GPU.  Nothing in simplyp_b200/ loads this library; the product has no CPU execution path.
#include <cmath>
#include <cstdint>

#include "../simplyp_b200/csrc/simplyp_ar1.cuh"

using namespace simplyp;

// The LOGLIK of one row as ar1_loglik_kernel forms it: observations o_row[D] (NaN: not observed), simulated values
// s_row[D], error scale em.  Day d is summed on lane d % 32 in day order, the 32 partial sums by the kernel's xor tree.
extern "C" double ar1_host_row(const double* o_row, const double* s_row, int D, double em, double phi) {
  double acc[32] = {0.0};
  double last_eta = 0.0;
  int last_day = -1;
  if (ar1_phi_valid(phi)) {
    for (int d0 = 0; d0 < D; d0 += 32) {
      double eta[32], sg[32], s[32];
      bool seen[32];
      for (int l = 0; l < 32; ++l) {
        const int d = d0 + l;
        const double o = d < D ? o_row[d] : NAN;
        seen[l] = o == o;
        s[l] = seen[l] ? s_row[d] : 1.0;
        eta[l] = ar1_eta(seen[l] ? o : 1.0, s[l], em, &sg[l]);
      }
      int prev = -1;
      for (int l = 0; l < 32; ++l) {
        if (!seen[l]) continue;
        const int pred = prev >= 0 ? d0 + prev : last_day;
        const double rho = pred < 0 ? 0.0 : ar1_rho(phi, d0 + l - pred);
        const double eta_prev = prev >= 0 ? eta[prev] : (pred < 0 ? 0.0 : last_eta);
        acc[l] = mc_add(acc[l], ar1_term(s[l], sg[l], eta[l], rho, eta_prev));
        prev = l;
      }
      if (prev >= 0) {
        last_eta = eta[prev];
        last_day = d0 + prev;
      }
    }
  }
  for (int off = 16; off > 0; off >>= 1) {
    double next[32];
    for (int l = 0; l < 32; ++l) next[l] = mc_add(acc[l], acc[l ^ off]);
    for (int l = 0; l < 32; ++l) acc[l] = next[l];
  }
  return ar1_finish(phi, acc[0]);
}

// The parameter-row writes of one member (what the propose, DE-trial and Sobol'-design kernels do with values[K]).
extern "C" void ar1_host_write_targets(const SimplypMcmcParam* param, int K, int S, const double* values, double* mrow,
                                       double* srow) {
  for (int i = 0; i < K; ++i) mcmc_write_target(param[i], S, values[i], mrow, srow);
}
