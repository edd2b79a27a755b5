// TEST HARNESS ONLY — compiles simplyp_core.cuh / simplyp_quad.cuh (and the scalar cross-check program, scalar_program.h) for the host so that the
// CPU-only test tier (`pytest -m "not gpu"`) can exercise the same per-thread arithmetic and
// control flow the CUDA kernels run, against the oracle, in a container without a GPU.
// Nothing in simplyp_b200/ loads this library; the product has no CPU execution path.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "scalar_program.h"
#include "../../simplyp_b200/csrc/simplyp_quad.cuh"
#include "../../simplyp_b200/csrc/simplyp_plan.cuh"

using namespace simplyp;

namespace {
struct HostIO {
  const double* fdata; const double* scp; const int32_t* po; const int32_t* pid;
  double* out; int S, D, m, s;

  void forcing(int day, double& P, double& E, double& doy) const {
    P = fdata[4 * day]; E = fdata[4 * day + 1]; doy = fdata[4 * day + 2];
  }
  void forcing(int day, double& P, double& E, double& doy, double& T_air) const {
    P = fdata[4 * day]; E = fdata[4 * day + 1]; doy = fdata[4 * day + 2]; T_air = fdata[4 * day + 3];
  }
  void upstream(int day, double (&us)[4]) const {
    us[0] = us[1] = us[2] = us[3] = 0.0;
    const double A_this = scp[(size_t)s * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
    for (int e = po[s]; e < po[s + 1]; ++e) {
      const int p = pid[e];
      const double* row = out + (((size_t)m * S + p) * D + day) * SIMPLYP_NOUT;
      const double A_up = scp[(size_t)p * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
      us[0] += row[SIMPLYP_O_QR] * (A_up / A_this);
      us[1] += row[SIMPLYP_O_MSUS_FLUX];
      us[2] += row[SIMPLYP_O_TDP_FLUX];
      us[3] += row[SIMPLYP_O_PP_FLUX];
    }
  }
  bool wants_vr() const { return true; }
  bool ready(int) const { return true; }
  void wait(int) const {}
  void publish(int) const {}
  static constexpr bool kAllLanesEmit = false;
  template <class Q>      // quad program: every lane calls it; the host's four lanes are one call
  void emit(const Q&, int day, const double (&y)[NL], double Vr, const double (&acc)[NA], const double (&non)[13],
            const Cold& c) const { emit(day, y, Vr, acc, non, c); }
  void emit(int day, const double (&y)[NL], double Vr, const double (&acc)[NA], const double (&non)[13],
            const Cold&) const {
    double* row = out + (((size_t)m * S + s) * D + day) * SIMPLYP_NOUT;
    row[0] = y[iVsA]; row[1] = y[iVsS]; row[2] = y[iVg]; row[3] = Vr; row[4] = y[iQr]; row[5] = acc[0];
    row[6] = y[iMsus]; row[7] = acc[1]; row[8] = y[iTDPr]; row[9] = acc[2]; row[10] = y[iPPr]; row[11] = acc[3];
    for (int i = 0; i < 13; ++i) row[12 + i] = non[i];
  }
};
}  // namespace

extern "C" int hostemu_run(const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                           const double* member_params, const double* sc_params, const int32_t* po,
                           const int32_t* pid, double* out, int64_t* diag) {
  const int M = dims->n_members, S = dims->n_sc, D = dims->n_days, Msc = dims->n_sc_param_sets;
  ThreadOptions t;
  t.rtol = opt->rtol; t.atol = opt->atol; t.step_len = opt->step_len;
  t.max_steps_per_day = opt->max_steps_per_day > 0 ? opt->max_steps_per_day : 5000;
  t.dynamic_epc0 = opt->dynamic_epc0; t.dynamic_erod = opt->dynamic_erodibility;
  t.run_mode_cal = opt->run_mode_cal; t.strict_quirks = opt->strict_quirks;
  t.snow_on_device = opt->snow_on_device;
  for (int m = 0; m < M; ++m) {
    const double* mp = member_params + (size_t)m * SIMPLYP_NP_MEMBER;
    const double* scp = sc_params + (size_t)(Msc > 1 ? m : 0) * S * SIMPLYP_NP_SC;
    const double* spl = scp + (size_t)(S - 1) * SIMPLYP_NP_SC;
    const double fNCA_last = spl[SIMPLYP_SC_F_AR] * spl[SIMPLYP_SC_F_NC_AR] + spl[SIMPLYP_SC_F_NC_IG] * spl[SIMPLYP_SC_F_IG];
    const int nc_last = fNCA_last > 0.0 ? 1 : (spl[SIMPLYP_SC_F_NC_S] > 0.0 ? 2 : 0);
    const double A_qr0 = scp[(size_t)opt->sc_qr0 * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
    for (int s = 0; s < S; ++s) {   // run order is upstream-first
      HostIO io{forcing, scp, po, pid, out, S, D, m, s};
      Cold c;
      ThreadCounters cnt;
      RegStages ks;
      run_member_sc(mp, scp + (size_t)s * SIMPLYP_NP_SC, A_qr0, nc_last, t, D, c, io, ks, cnt);
      if (diag) {
        int64_t* dg = diag + ((size_t)m * S + s) * SIMPLYP_NDIAG;
        dg[0] = cnt.steps; dg[1] = cnt.rejected; dg[2] = cnt.rhs_evals; dg[3] = cnt.status;
      }
    }
  }
  return 0;
}



// The quad program (simplyp_quad.cuh) executed with the 4 lanes as the 4 elements of a struct.
extern "C" int hostemu_run_quad(const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                                const double* member_params, const double* sc_params, const int32_t* po,
                                const int32_t* pid, double* out, int64_t* diag) {
  const int M = dims->n_members, S = dims->n_sc, D = dims->n_days, Msc = dims->n_sc_param_sets;
  ThreadOptions t;
  t.rtol = opt->rtol; t.atol = opt->atol; t.step_len = opt->step_len;
  t.max_steps_per_day = opt->max_steps_per_day > 0 ? opt->max_steps_per_day : 5000;
  t.dynamic_epc0 = opt->dynamic_epc0; t.dynamic_erod = opt->dynamic_erodibility;
  t.run_mode_cal = opt->run_mode_cal; t.strict_quirks = opt->strict_quirks;
  t.snow_on_device = opt->snow_on_device;
  for (int m = 0; m < M; ++m) {
    const double* mp = member_params + (size_t)m * SIMPLYP_NP_MEMBER;
    const double* scp = sc_params + (size_t)(Msc > 1 ? m : 0) * S * SIMPLYP_NP_SC;
    const double* spl = scp + (size_t)(S - 1) * SIMPLYP_NP_SC;
    const double fNCA_last = spl[SIMPLYP_SC_F_AR] * spl[SIMPLYP_SC_F_NC_AR] + spl[SIMPLYP_SC_F_NC_IG] * spl[SIMPLYP_SC_F_IG];
    const int nc_last = fNCA_last > 0.0 ? 1 : (spl[SIMPLYP_SC_F_NC_S] > 0.0 ? 2 : 0);
    const double A_qr0 = scp[(size_t)opt->sc_qr0 * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
    for (int s = 0; s < S; ++s) {
      HostIO io{forcing, scp, po, pid, out, S, D, m, s};
      QuadHost4 q;
      QuadMem qm;
      ThreadCounters cnt;
      run_quad<true>(q, mp, scp + (size_t)s * SIMPLYP_NP_SC, A_qr0, nc_last, t, D, true, qm, io, cnt);
      if (diag) {
        int64_t* dg = diag + ((size_t)m * S + s) * SIMPLYP_NDIAG;
        dg[0] = cnt.steps; dg[1] = cnt.rejected; dg[2] = cnt.rhs_evals; dg[3] = cnt.status;
      }
    }
  }
  return 0;
}

// One sub-catchment, the record integrated in two launches' worth of pieces: days [0, split) with the midnight state
// stored (what the cost pilot does), then days [split, D) continued from it (what the main launch does).
extern "C" int hostemu_run_quad_split(const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                                      const double* member_params, const double* sc_params, const int32_t* po,
                                      const int32_t* pid, double* out, int64_t* diag, int split) {
  const int M = dims->n_members, S = dims->n_sc, D = dims->n_days, Msc = dims->n_sc_param_sets;
  if (S != 1 || split <= 0 || split >= D) return -1;
  ThreadOptions t;
  t.rtol = opt->rtol; t.atol = opt->atol; t.step_len = opt->step_len;
  t.max_steps_per_day = opt->max_steps_per_day > 0 ? opt->max_steps_per_day : 5000;
  t.dynamic_epc0 = opt->dynamic_epc0; t.dynamic_erod = opt->dynamic_erodibility;
  t.run_mode_cal = opt->run_mode_cal; t.strict_quirks = opt->strict_quirks;
  t.snow_on_device = opt->snow_on_device;
  std::vector<QuadCarry> carry(M);
  for (int pass = 0; pass < 2; ++pass)
    for (int m = 0; m < M; ++m) {
      const double* mp = member_params + (size_t)m * SIMPLYP_NP_MEMBER;
      const double* scp = sc_params + (size_t)(Msc > 1 ? m : 0) * SIMPLYP_NP_SC;
      const double fNCA_last = scp[SIMPLYP_SC_F_AR] * scp[SIMPLYP_SC_F_NC_AR] + scp[SIMPLYP_SC_F_NC_IG] * scp[SIMPLYP_SC_F_IG];
      const int nc_last = fNCA_last > 0.0 ? 1 : (scp[SIMPLYP_SC_F_NC_S] > 0.0 ? 2 : 0);
      HostIO io{forcing, scp, po, pid, out, 1, D, m, 0};
      QuadHost4 q;
      QuadMem qm;
      ThreadCounters cnt;
      if (pass == 0) run_quad<true>(q, mp, scp, scp[SIMPLYP_SC_A_CATCH], nc_last, t, split, true, qm, io, cnt, 0, nullptr, &carry[m]);
      else run_quad<true>(q, mp, scp, scp[SIMPLYP_SC_A_CATCH], nc_last, t, D, true, qm, io, cnt, split, &carry[m], nullptr);
      if (diag && pass == 1) {
        int64_t* dg = diag + (size_t)m * SIMPLYP_NDIAG;
        dg[0] = cnt.steps; dg[1] = cnt.rejected; dg[2] = cnt.rhs_evals; dg[3] = cnt.status;
      }
    }
  return 0;
}

// Placement plan arithmetic (simplyp_plan.cuh) for M members on n_sm SMs: item index of every cost rank, and for
// every virtual block the list that runs it and its position in that list.  Returns 0 if the plan does not apply.
extern "C" int hostemu_plan(int M, int n_sm, int solo, int resident, int* index_of_rank, int* list_of_block,
                            int* pos_in_list, int* shape6) {
  PlanShape p;
  const long long B = ((long long)M + 31) / 32;
  if (!plan_shape(B, n_sm, p, resident)) return 0;
  shape6[0] = p.nY; shape6[1] = p.nP; shape6[2] = p.Q; shape6[3] = p.n_lists(); shape6[4] = p.n_launch();
  shape6[5] = p.resident;
  const MemberLayout L = member_layout(p, M, solo);
  for (int r = 0; r < M; ++r) index_of_rank[r] = member_layout_index(r, L);
  for (int b = 0; b < (int)B; ++b) { list_of_block[b] = -1; pos_in_list[b] = -1; }
  for (int l = 0; l < 3 * n_sm; ++l) {
    int pos = 0;
    for (int vb = plan_list_head(p, l); vb >= 0; vb = plan_list_next(p, vb), ++pos) {
      if (vb >= (int)B || list_of_block[vb] != -1) return -1;      // out of range or claimed twice
      list_of_block[vb] = l; pos_in_list[vb] = pos;
    }
  }
  return 1;
}

// Launch policy of the quad kernel (simplyp_plan.cuh) under the overrides in the environment.  out[12]: grid, minb,
// pilot_days, pilot_minb, plan, nY, nP, Q, resident, solo, epoch_days, n_epochs.
extern "C" void hostemu_launch_config(int M, int D, int network, int n_levels, long long grid_one_epoch, int pilot_days,
                                      int workspace, int n_sm, long long* out) {
  const LaunchInputs in = {M, D, network != 0, n_levels, grid_one_epoch, pilot_days, workspace != 0, n_sm};
  const LaunchConfig c = launch_config(in, read_launch_overrides());
  const long long v[12] = {c.grid, c.minb, c.pilot_days, c.pilot_minb, c.plan, c.shape.nY, c.shape.nP, c.shape.Q,
                           c.shape.resident, c.solo, c.epoch_days, c.n_epochs};
  memcpy(out, v, sizeof(v));
}

// The quad formulation of ode_f against the scalar rhs() at one state: returns the largest relative
// difference over the 12 derivatives (dQr/dt and dVr/dt are recovered from du/dt and the quad's slot B).
extern "C" double hostemu_quad_rhs_check(const double* mp, const double* sp, double P, double E, double doy,
                                         const double* us4, const double* y7, int dynamic_epc0, int dynamic_erod) {
  Hot h; Cold c; Flags fl; DayAux aux; double y0[NL], Kf;
  setup_thread(mp, sp, sp[SIMPLYP_SC_A_CATCH], 0, 1, 1, h, c, fl, y0, Kf);
  double us[4] = {us4[0], us4[1], us4[2], us4[3]};
  begin_day(mp, sp, c, fl, dynamic_epc0, dynamic_erod, P, E, doy, us, h, aux);
  double y[NL], dy[NL], da[NA];
  for (int i = 0; i < NL; ++i) y[i] = y7[i];
  rhs(h, y, dy, da);
  QuadHost4 q;
  QuadCoef<QuadHost4> qc;
  quad_static_coef(q, h, qc);
  quad_daily_coef(q, h, qc);
  const double Qr = y[iQr], Vr = reach_volume(h, Qr);
  const V4 yA = q.pick(y[iVsA], y[iVsS], y[iVg], log(Qr));
  const V4 yB = q.pick(y[iMsus], y[iTDPr], y[iPPr], Vr);
  V4 dA, dB, dacc, e;
  quad_rhs(q, qc, yA, yB, dA, dB, dacc, e);
  const double got[12] = {dA.v[0], dA.v[1], dA.v[2], dA.v[3] * Qr, dB.v[0], dB.v[1], dB.v[2],
                          dacc.v[3], dacc.v[0], dacc.v[1], dacc.v[2], dB.v[3]};
  // ode_f's dVr/dt = net = dQr/dt / (kQ Qr^b_Q) (:127-131)
  const double net = dy[iQr] / (h.kQ * exp(h.bQ * log(Qr)));
  const double want[12] = {dy[iVsA], dy[iVsS], dy[iVg], dy[iQr], dy[iMsus], dy[iTDPr], dy[iPPr],
                           da[0], da[1], da[2], da[3], net};
  double worst = 0.0;
  for (int i = 0; i < 12; ++i) {
    const double scale = fmax(fabs(want[i]), 1e-12 * (1.0 + fabs(y[i < NL ? i : 0])));
    worst = fmax(worst, fabs(got[i] - want[i]) / scale);
  }
  return worst;
}

extern "C" void hostemu_exp_tab(const double* x, double* y, int n) {
  for (int i = 0; i < n; ++i) y[i] = sp_exp_tab(x[i], kExp2Tab);
}
