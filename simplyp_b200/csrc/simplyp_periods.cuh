// simplyp_periods.cuh — arithmetic of the receiving water body (waterbody_kernel) and of the period aggregates of an
// ensemble (period_aggregate_kernel; simplyp_period_aggregates_device, include/simplyp_b200.h).
//
// One day of sum_to_waterbody (model.py:851-900): over the reaches flagged In_final_flux? == 1, in their order,
// q += Qr*A*1000/86400 (Q_cumecs, :784) and the Msus / TDP / PP daily fluxes are summed; the concentrations are
// (flux/q)*(1000/86400) (:889-892) and TP, SRP follow as in derived_P_species (:831-847).  The expressions are
// written once, over an arithmetic policy P:
//   WbPlain   plain operators, as waterbody_kernel has always been compiled.  Its SASS has no DFMA in them: every sum
//             adds a quotient or a column, and TP_mgl is a DADD of the two stored concentrations.
//   WbRounded every operation rounded on its own (mc_*), for the period aggregates: whatever the context, nothing can
//             be contracted, so the host build (g++ -ffp-contract=off) gives the same bits.
// Both give the same IEEE operations in the same order.
//
// The period aggregates.  A series is (target, kind, statistic): target a run-order reach, or PERIOD_WATERBODY for the
// flagged reaches; kind a SIMPLYP_V_* kind; statistic
//   PERIOD_MEAN  sum over the period's days of the daily value, divided by the number of days; the daily value of a
//                reach is sim_series_value (what the fit statistics and the bands see), of the water body the
//                concentration or Q_cumecs of sum_to_waterbody;
//   PERIOD_LOAD  sum of the daily flux in kg (Q: the volume in m3, Q_cumecs*86400; TP = TDP + PP; SRP = f_TDP*TDP);
//   PERIOD_FWMC  (sum of the flux / sum of Q_cumecs)*(1000/86400), undefined for Q.
// The flux and Q_cumecs of a reach are those of a water body made of that one reach.  Every sum runs over the days in
// ascending order, one rounding per addition, starting from 0.
//
// Inline __host__ __device__ code like simplyp_bands.cuh: the CPU test tier compiles it for the host.
#pragma once

#include "simplyp_bands.cuh"

namespace simplyp {

struct WbPlain {
  static SP_HD double add(double a, double b) { return a + b; }
  static SP_HD double mul(double a, double b) { return a * b; }
  static SP_HD double div(double a, double b) { return a / b; }
};
struct WbRounded {
  static SP_HD double add(double a, double b) { return mc_add(a, b); }
  static SP_HD double mul(double a, double b) { return mc_mul(a, b); }
  static SP_HD double div(double a, double b) { return mc_div(a, b); }
};

// Daily sums of the water body: adds one reach's row of the raw output; sc = the reach's row of sc_params.  (The
// A_catch load follows the Qr load, as it always has in waterbody_kernel.)
template <class P>
SP_HD void wb_add_reach(const double* row, const double* sc, double& q, double& ms, double& td, double& pp) {
  q = P::add(q, P::div(P::mul(P::mul(row[SIMPLYP_O_QR], sc[SIMPLYP_SC_A_CATCH]), 1000.0), 86400.0));
  ms = P::add(ms, row[SIMPLYP_O_MSUS_FLUX]);
  td = P::add(td, row[SIMPLYP_O_TDP_FLUX]);
  pp = P::add(pp, row[SIMPLYP_O_PP_FLUX]);
}

// Concentration in mg/l of a flux in kg/day (or of a sum of them) carried by Q_cumecs q (or by their sum).
template <class P>
SP_HD double wb_conc(double flux, double q) { return P::mul(P::div(flux, q), 1000.0 / 86400.0); }

// The SIMPLYP_NWB columns of one day (Engine.WATERBODY_COLUMNS).
template <class P>
SP_HD void wb_columns(double q, double ms, double td, double pp, double f_TDP, double* w) {
  const double ss_mgl = wb_conc<P>(ms, q), tdp_mgl = wb_conc<P>(td, q), pp_mgl = wb_conc<P>(pp, q);
  w[0] = q; w[1] = ms; w[2] = td; w[3] = pp; w[4] = ss_mgl; w[5] = tdp_mgl; w[6] = pp_mgl;
  w[7] = P::add(tdp_mgl, pp_mgl);      // TP_mgl    (:842)
  w[8] = P::add(td, pp);               // TP_kg/day (:843)
  w[9] = P::mul(tdp_mgl, f_TDP);       // SRP_mgl   (:844)
  w[10] = P::mul(td, f_TDP);           // SRP_kg/day (:845)
}

// The daily value of a kind in the water body: the column of wb_columns that Q_cumecs or the concentration is.
template <class P>
SP_HD double wb_value(int kind, double q, double ms, double td, double pp, double f_TDP) {
  switch (kind) {
    case SIMPLYP_V_Q:   return q;
    case SIMPLYP_V_SS:  return wb_conc<P>(ms, q);
    case SIMPLYP_V_TDP: return wb_conc<P>(td, q);
    case SIMPLYP_V_PP:  return wb_conc<P>(pp, q);
    case SIMPLYP_V_TP:  return P::add(wb_conc<P>(td, q), wb_conc<P>(pp, q));
    default:            return P::mul(wb_conc<P>(td, q), f_TDP);
  }
}

constexpr int PERIOD_MEAN = SIMPLYP_PERIOD_MEAN, PERIOD_LOAD = SIMPLYP_PERIOD_LOAD, PERIOD_FWMC = SIMPLYP_PERIOD_FWMC;
constexpr int PERIOD_WATERBODY = SIMPLYP_PERIOD_WATERBODY;

// The daily flux of a kind in kg (m3 for Q): Q_cumecs*86400, or the column of wb_columns.
SP_HD double period_flux(int kind, double q, double ms, double td, double pp, double f_TDP) {
  switch (kind) {
    case SIMPLYP_V_Q:   return mc_mul(q, 86400.0);
    case SIMPLYP_V_SS:  return ms;
    case SIMPLYP_V_TDP: return td;
    case SIMPLYP_V_PP:  return pp;
    case SIMPLYP_V_TP:  return mc_add(td, pp);
    default:            return mc_mul(td, f_TDP);
  }
}

// One (member, day) of a series: x = the daily value (PERIOD_MEAN) or flux, q = Q_cumecs (PERIOD_FWMC; else 0).
// out_m [S][D][NOUT] and scp_m [S][NP_SC] are the member's output and sub-catchment rows, wb[n_wb] the run-order
// reaches of the water body.
SP_HD void period_day(const double* out_m, const double* scp_m, double f_TDP, int D, int d, int target, int kind,
                      int stat, const int* wb, int n_wb, double* x, double* q) {
  if (stat == PERIOD_MEAN && target != PERIOD_WATERBODY) {
    const double* row = out_m + ((size_t)target * D + d) * SIMPLYP_NOUT;
    const double A = scp_m[(size_t)target * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
    const double Qr = row[SIMPLYP_O_QR];
    *x = sim_series_value(kind, Qr, row[SIMPLYP_O_MSUS_FLUX], row[SIMPLYP_O_TDP_FLUX], row[SIMPLYP_O_PP_FLUX], A,
                          sp_rcp(Qr), sp_rcp(A), f_TDP);
    *q = 0.0;
    return;
  }
  double qs = 0.0, ms = 0.0, td = 0.0, pp = 0.0;
  const int n = target == PERIOD_WATERBODY ? n_wb : 1;
  for (int k = 0; k < n; ++k) {
    const int s = target == PERIOD_WATERBODY ? wb[k] : target;
    wb_add_reach<WbRounded>(out_m + ((size_t)s * D + d) * SIMPLYP_NOUT, scp_m + (size_t)s * SIMPLYP_NP_SC, qs, ms, td,
                            pp);
  }
  *x = stat == PERIOD_MEAN ? wb_value<WbRounded>(kind, qs, ms, td, pp, f_TDP)
                           : period_flux(kind, qs, ms, td, pp, f_TDP);
  *q = stat == PERIOD_FWMC ? qs : 0.0;
}

// The aggregate of a period of n_days days from the day-ordered sums of x and q.
SP_HD double period_result(int stat, double sx, double sq, int n_days) {
  switch (stat) {
    case PERIOD_MEAN: return mc_div(sx, (double)n_days);
    case PERIOD_LOAD: return sx;
    default:          return wb_conc<WbRounded>(sx, sq);
  }
}

}  // namespace simplyp
