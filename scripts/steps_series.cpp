// Analysis tool: daily output series + attempt counts of the quad program on the host under run-time error-norm weights
// (error-norm experiments).   g++ -O2 -fopenmp -std=c++17 -shared -fPIC -o build/libsteps_series.so scripts/steps_series.cpp
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
static double g_wB = 1.0, g_wACC = 1.0, g_wU = 1.0, g_wVG = 1.0, g_wSOIL = 1000.0;
#define SP_W_B g_wB
#define SP_W_ACC g_wACC
#define SP_W_U g_wU
#define SP_W_VG g_wVG
#define SP_SOIL_ERR_WEIGHT g_wSOIL
#include "../simplyp_b200/csrc/simplyp_quad.cuh"
using namespace simplyp;
struct IO {
  const double* f; double* out; int D;
  void wait(int) const {}
  void forcing(int day, double& P, double& E, double& doy, double& T) const { P = f[4*day]; E = f[4*day+1]; doy = f[4*day+2]; T = f[4*day+3]; }
  void upstream(int, double (&us)[4]) const { us[0]=us[1]=us[2]=us[3]=0; }
  void publish(int) const {}
  template <class Q> void emit(const Q&, int day, const double (&y)[NL], double Vr, const double (&acc)[NA], const double (&)[13], const Cold&) {
    double* o = out + (size_t)day * 12;
    for (int i = 0; i < 4; ++i) o[i] = acc[i];
    for (int i = 0; i < NL; ++i) o[4 + i] = y[i];
    o[11] = Vr;
  }
};
extern "C" int steps_series(int M, int D, const double* forcing, const double* mp, const double* scp, double rtol, double atol,
                            const double* w, long long* steps, long long* rej, double* out) {
  g_wB = w[0]; g_wACC = w[1]; g_wU = w[2]; g_wVG = w[3]; g_wSOIL = w[4];
  ThreadOptions t; memset(&t, 0, sizeof(t)); t.rtol = rtol; t.atol = atol; t.step_len = 1.0; t.max_steps_per_day = 5000;
  t.dynamic_epc0 = 1; t.dynamic_erod = 1; t.run_mode_cal = 1; t.strict_quirks = 1;
#pragma omp parallel for schedule(dynamic, 8)
  for (int m = 0; m < M; ++m) {
    ThreadCounters cnt; QuadMem qm; QuadHost4 q; IO io{forcing, out + (size_t)m * D * 12, D};
    run_quad<false>(q, mp + (size_t)m * SIMPLYP_NP_MEMBER, scp, scp[SIMPLYP_SC_A_CATCH], 0, t, D, true, qm, io, cnt);
    steps[m] = cnt.steps; rej[m] = cnt.rejected;
  }
  return 0;
}
