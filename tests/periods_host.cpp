// TEST HARNESS ONLY — compiles simplyp_periods.cuh (the water body's daily sums and the period aggregates) for the
// host, so that the CPU-only test tier can check it against NumPy without a GPU.  Nothing in simplyp_b200/ loads this
// library; the product has no CPU execution path.
#include <cmath>
#include <cstdint>

#include "../simplyp_b200/csrc/simplyp_periods.cuh"

using namespace simplyp;

// waterbody_kernel's columns wb[M][D][SIMPLYP_NWB] from out[M][S][D][25], sc_params[Msc][S][NP_SC],
// member_params[M][NP_MEMBER] and the run-order reaches[n].
extern "C" void periods_host_waterbody(const double* out, const double* sc_params, const double* member_params,
                                       const int32_t* reaches, int n, int M, int S, int D, int Msc, double* wb) {
  for (int m = 0; m < M; ++m)
    for (int d = 0; d < D; ++d) {
      const double* scp = sc_params + (size_t)(Msc > 1 ? m : 0) * S * SIMPLYP_NP_SC;
      double q = 0.0, ms = 0.0, td = 0.0, pp = 0.0;
      for (int k = 0; k < n; ++k)
        wb_add_reach<WbPlain>(out + (((size_t)m * S + reaches[k]) * D + d) * SIMPLYP_NOUT,
                              scp + (size_t)reaches[k] * SIMPLYP_NP_SC, q, ms, td, pp);
      wb_columns<WbPlain>(q, ms, td, pp, member_params[(size_t)m * SIMPLYP_NP_MEMBER + SIMPLYP_P_F_TDP],
                          wb + ((size_t)m * D + d) * SIMPLYP_NWB);
    }
}

// What period_aggregate_kernel writes for a chunk of M members: values[V * P][M] (member_offset 0, M_total = M).
extern "C" void periods_host_aggregate(const double* out, const double* member_params, const double* sc_params,
                                       const int64_t* diag, const int32_t* series, int V, const int32_t* bounds, int P,
                                       const int32_t* wb, int n_wb, int M, int S, int D, int Msc, double* values) {
  for (int m = 0; m < M; ++m) {
    int failed = 0;
    for (int r = 0; r < S; ++r) failed |= diag[((size_t)m * S + r) * SIMPLYP_NDIAG + SIMPLYP_DG_STATUS] != 0;
    const double* out_m = out + (size_t)m * S * D * SIMPLYP_NOUT;
    const double* scp = sc_params + (size_t)(Msc > 1 ? m : 0) * S * SIMPLYP_NP_SC;
    const double f_TDP = member_params[(size_t)m * SIMPLYP_NP_MEMBER + SIMPLYP_P_F_TDP];
    for (int v = 0; v < V; ++v)
      for (int p = 0; p < P; ++p) {
        double res = NAN;
        if (!failed) {
          double sx = 0.0, sq = 0.0;
          for (int d = bounds[2 * p]; d <= bounds[2 * p + 1]; ++d) {
            double x, q;
            period_day(out_m, scp, f_TDP, D, d, series[3 * v], series[3 * v + 1], series[3 * v + 2], wb, n_wb, &x, &q);
            sx = mc_add(sx, x);
            sq = mc_add(sq, q);
          }
          res = period_result(series[3 * v + 2], sx, sq, bounds[2 * p + 1] - bounds[2 * p] + 1);
        }
        values[((size_t)v * P + p) * M + m] = res;
      }
  }
}
