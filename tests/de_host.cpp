// TEST HARNESS ONLY — compiles simplyp_de.cuh (the per-member arithmetic of differential evolution: picks, trials,
// scaling, energies, selection) for the host, so that the CPU-only test tier can check it against the NumPy
// restatement (tests/de_reference.py) without a GPU.  Nothing in simplyp_b200/ loads this library; the product has no
// CPU execution path.
#include <cmath>
#include <cstdint>

#include "../simplyp_b200/csrc/simplyp_de.cuh"

using namespace simplyp;

// The mutation factor of generation g.
extern "C" double de_host_dither(const SimplypDe* de, long long g) { return de_dither(*de, g); }

// Picks and fill point of every member at generation g: out[N][4] = (r0, r1, r2 or -1, fill).
extern "C" void de_host_picks(const SimplypDe* de, long long g, int32_t* out) {
  for (int i = 0; i < de->n_population; ++i) {
    int r[3], fill;
    de_picks(*de, g, i, r, &fill);
    for (int q = 0; q < 3; ++q) out[4 * i + q] = r[q];
    out[4 * i + 3] = fill;
  }
}

// Trials of every member at generation g (what de_trial_kernel computes): trial[N][K] from pop[N][K].
extern "C" void de_host_trials(const SimplypDe* de, const double* pop, long long best, long long g, double* trial) {
  const double F = de_dither(*de, g);
  for (int i = 0; i < de->n_population; ++i)
    de_trial_member(*de, pop, best, g, i, F, trial + (size_t)i * de->n_free);
}

// Parameter values of unit-cube rows u[n][K]: out[n][K].
extern "C" void de_host_scale(const SimplypDe* de, long long n, const double* u, double* out) {
  const int K = de->n_free;
  for (long long m = 0; m < n; ++m)
    for (int j = 0; j < K; ++j) out[m * K + j] = de_scale(de->param[j], u[m * K + j]);
}

// Energies of N members from y[R][N], w[R] and diag[N][S][SIMPLYP_NDIAG]: out[N].
extern "C" void de_host_energy(const double* y, long long N, int R, const double* w, const int64_t* diag, int S,
                               double* out) {
  for (long long m = 0; m < N; ++m) out[m] = de_energy(y, N, R, w, m, diag + (size_t)m * S * SIMPLYP_NDIAG, S);
}

// Selection of every member (what de_select_kernel does after de_energy); replaced[N] = 1 where the trial won.
extern "C" void de_host_select(int K, int N, const double* e_trial, const double* trial, double* pop, double* energy,
                               int32_t* replaced) {
  for (int i = 0; i < N; ++i) replaced[i] = de_select_member(K, i, e_trial[i], trial + (size_t)i * K, pop, energy);
}
