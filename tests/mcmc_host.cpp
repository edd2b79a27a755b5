// TEST HARNESS ONLY — compiles simplyp_mcmc.cuh (the ensemble sampler's per-walker arithmetic) for the host so that
// the CPU-only test tier can check it against the NumPy reference sampler (tests/mcmc_reference.py) without a GPU.
// Nothing in simplyp_b200/ loads this library; the product has no CPU execution path.
#include <cmath>
#include <cstdint>

#include "../simplyp_b200/csrc/simplyp_mcmc.cuh"

using namespace simplyp;

// Philox4x32-10: n counters ctr[n][4] under keys key[n][2] -> out[n][4].
extern "C" void mcmc_host_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out, int n) {
  for (int i = 0; i < n; ++i) {
    const uint32_t c[4] = {ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3]};
    uint32_t r[4];
    philox4x32_10(c, key[2 * i], key[2 * i + 1], r);
    for (int j = 0; j < 4; ++j) out[4 * i + j] = r[j];
  }
}

// The proposals of every walker of one half (what mcmc_propose_kernel computes): prop[W/2][K], log_z[W/2], flags.
extern "C" void mcmc_host_propose(const SimplypMcmc* mc, const double* walkers, long long t, int half, double* prop,
                                  double* log_z, int32_t* out_of_box) {
  const int H = mc->n_walkers / 2;
  for (int k = 0; k < H; ++k)
    out_of_box[k] = mcmc_propose_walker(*mc, walkers, t, half, k, prop + (size_t)k * mc->n_free, log_z + k);
}

// The Metropolis-Hastings step of every walker of one half given the proposals' log-probabilities lp_new[W/2]
// (what mcmc_accept_kernel does after mcmc_member_lp); decisions[W/2] = 1 where accepted.
extern "C" void mcmc_host_accept(const SimplypMcmc* mc, long long t, int half, const double* lp_new,
                                 const double* log_z, const double* prop, double* walkers, double* lp,
                                 int64_t* accepted, int32_t* decisions) {
  const int H = mc->n_walkers / 2;
  for (int k = 0; k < H; ++k)
    decisions[k] = mcmc_accept_walker(*mc, t, half, k, lp_new[k], log_z[k], prop + (size_t)k * mc->n_free, walkers,
                                      lp, accepted);
}
