// TEST HARNESS ONLY — compiles simplyp_nsga2.cuh (the per-pair arithmetic of NSGA-II: tournaments, SBX, polynomial
// mutation, orientation, dominance) for the host, so that the CPU-only test tier can check it against the NumPy
// restatement (tests/nsga2_reference.py) without a GPU.  Nothing in simplyp_b200/ loads this library; the product has
// no CPU execution path.
#include <cmath>
#include <cstdint>

#include "../simplyp_b200/csrc/simplyp_nsga2.cuh"

using namespace simplyp;

// Tournament picks of every pair at generation g: out[N/2][4].
extern "C" void nsga2_host_picks(const SimplypNsga2* ns, long long g, int32_t* out) {
  for (int p = 0; p < ns->n_population / 2; ++p) {
    int picks[4];
    nsga2_picks(*ns, g, p, picks);
    for (int t = 0; t < 4; ++t) out[4 * p + t] = picks[t];
  }
}

// Offspring of every pair at generation g (what nsga2_offspring_kernel computes): children[N][K], dec[N/2][3 + K].
extern "C" void nsga2_host_offspring(const SimplypNsga2* ns, const double* pop, const int32_t* rank,
                                     const double* crowd, long long g, double* children, int32_t* dec) {
  const int K = ns->n_free;
  for (int p = 0; p < ns->n_population / 2; ++p)
    nsga2_offspring_pair(*ns, pop, rank, crowd, g, p, children + (size_t)(2 * p) * K,
                         children + (size_t)(2 * p + 1) * K, dec + (size_t)p * (3 + K));
}

// Oriented objectives f[n][M] of y[M][n] with status[n]: what nsga2_load_kernel writes.
extern "C" void nsga2_host_orient(const SimplypNsga2* ns, const double* y, long long n, const int32_t* status,
                                  double* f) {
  for (long long i = 0; i < n; ++i) nsga2_orient(*ns, y + i, n, status[i], f + i * ns->n_objectives);
}

// dom[n][n]: dom[j * n + i] = 1 when row j of f[n][M] dominates row i.
extern "C" void nsga2_host_dominance(const double* f, long long n, int M, int32_t* dom) {
  for (long long j = 0; j < n; ++j)
    for (long long i = 0; i < n; ++i) dom[j * n + i] = nsga2_dominates(f + j * M, f + i * M, M);
}
