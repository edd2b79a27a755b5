// Analysis tool: total step attempts / rejections of the quad program per member (controller experiments).
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include "../simplyp_b200/csrc/simplyp_quad.cuh"
using namespace simplyp;
struct IO {
  const double* f;
  void wait(int) const {}
  void forcing(int day, double& P, double& E, double& doy, double& T) const { P = f[4*day]; E = f[4*day+1]; doy = f[4*day+2]; T = f[4*day+3]; }
  void upstream(int, double (&us)[4]) const { us[0]=us[1]=us[2]=us[3]=0; }
  bool wants_vr() const { return false; }
  void publish(int) const {}
  template <class Q> void emit(const Q&, int, const double (&)[NL], double, const double (&acc)[NA], const double (&)[13], const Cold&) { chk += acc[0]; }
  double chk = 0;
};
extern "C" int steps_quad(int M, int D, const double* forcing, const double* mp, const double* scp, double rtol, double atol,
                          long long* steps, long long* rej, double* chk) {
  ThreadOptions t; memset(&t, 0, sizeof(t)); t.rtol = rtol; t.atol = atol; t.step_len = 1.0; t.max_steps_per_day = 5000;
  t.dynamic_epc0 = 1; t.dynamic_erod = 1; t.run_mode_cal = 1; t.strict_quirks = 1;
#pragma omp parallel for schedule(dynamic, 16)
  for (int m = 0; m < M; ++m) {
    ThreadCounters cnt; QuadMem qm; QuadHost4 q; IO io{forcing};
    run_quad<false>(q, mp + (size_t)m * SIMPLYP_NP_MEMBER, scp, scp[SIMPLYP_SC_A_CATCH], 0, t, D, true, qm, io, cnt);
    steps[m] = cnt.steps; rej[m] = cnt.rejected; chk[m] = io.chk;
  }
  return 0;
}
