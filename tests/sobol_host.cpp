// TEST HARNESS ONLY — compiles simplyp_sobol.cuh (the direction numbers, Sobol' points, Saltelli design values and
// bootstrap picks of the sensitivity analysis) for the host, so that the CPU-only test tier can check it against
// SciPy and NumPy without a GPU.  Nothing in simplyp_b200/ loads this library; the product has no CPU execution path.
#include <cmath>
#include <cstdint>

#include "../simplyp_b200/csrc/simplyp_sobol.cuh"

using namespace simplyp;

// The embedded direction numbers: out[SOBOL_DIMS][32].
extern "C" void sobol_host_table(uint32_t* out) {
  for (int d = 0; d < SOBOL_DIMS; ++d)
    for (int j = 0; j < SOBOL_BITS; ++j) out[d * SOBOL_BITS + j] = sobol_v(d, j);
}

// Points skip .. skip + n - 1 of the D-dimensional sequence: out[n][D].
extern "C" void sobol_host_points(int D, int64_t n, int64_t skip, uint32_t* out) {
  for (int64_t i = 0; i < n; ++i)
    for (int d = 0; d < D; ++d) out[i * D + d] = sobol_coord(d, (uint32_t)(skip + i));
}

// Values of the K free parameters of design members member_offset .. member_offset + n - 1: out[n][K].
extern "C" void sobol_host_design(const SimplypSobol* sb, int64_t member_offset, int64_t n, double* out) {
  for (int64_t m = 0; m < n; ++m)
    for (int j = 0; j < sb->n_free; ++j) out[m * sb->n_free + j] = sobol_design_value(*sb, member_offset + m, j);
}

// Positions (in n used samples) of the draws 0 .. count - 1 of bootstrap resample t: out[count].
extern "C" void sobol_host_picks(uint64_t seed, uint32_t t, uint32_t n, int64_t count, uint32_t* out) {
  for (int64_t k = 0; k < count; k += 4) {
    uint32_t r[4];
    sobol_boot_words(seed, t, (uint32_t)(k / 4), r);
    for (int q = 0; q < 4 && k + q < count; ++q) out[k + q] = sobol_boot_pick(r[q], n);
  }
}
