// TEST HARNESS ONLY — compiles simplyp_bands.cuh (the error draws and the np.nanquantile index / interpolation
// arithmetic of the posterior predictive bands) for the host, so that the CPU-only test tier can check it against
// NumPy without a GPU.  Nothing in simplyp_b200/ loads this library; the product has no CPU execution path.
#include <cmath>
#include <cstdint>

#include "../simplyp_b200/csrc/simplyp_bands.cuh"

using namespace simplyp;

// The Philox words of the error draw of (member[i], day[i], series[i]) under `seed` -> out[n][4].
extern "C" void bands_host_words(uint64_t seed, const int32_t* member, const int32_t* day, const int32_t* series,
                                 uint32_t* out, int n) {
  for (int i = 0; i < n; ++i) {
    uint32_t r[4];
    band_words(seed, member[i], day[i], series[i], r);
    for (int j = 0; j < 4; ++j) out[4 * i + j] = r[j];
  }
}

// eps of (member[i], day[i], series[i]) under `seed`.
extern "C" void bands_host_epsilon(uint64_t seed, const int32_t* member, const int32_t* day, const int32_t* series,
                                   double* eps, int n) {
  for (int i = 0; i < n; ++i) eps[i] = band_epsilon(seed, member[i], day[i], series[i]);
}

// The quantiles of q[n_q] of every row of sorted[R][N] (ascending, NaN last) with n[r] non-NaN entries, as the
// selection kernels form them from the order statistics: out[n_q][R].
extern "C" void bands_host_quantiles(const double* sorted, const int64_t* n, int64_t R, int64_t N, const double* q,
                                     int n_q, double* out) {
  for (int64_t r = 0; r < R; ++r)
    for (int k = 0; k < n_q; ++k) {
      double res = NAN;
      if (n[r] > 0) {
        long long lo, hi;
        double g;
        nq_index(n[r], q[k], &lo, &hi, &g);
        res = nq_lerp(sorted[r * N + lo], sorted[r * N + hi], g);
      }
      out[k * R + r] = res;
    }
}

// Order-preserving keys of x[n] and back.
extern "C" void bands_host_keys(const double* x, uint64_t* keys, double* back, int64_t n) {
  for (int64_t i = 0; i < n; ++i) {
    keys[i] = nq_key(x[i]);
    back[i] = nq_value(keys[i]);
  }
}
