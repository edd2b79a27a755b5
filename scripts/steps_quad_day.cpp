// Analysis tool: per-member per-day step attempts of the quad program on the host (SP_DAY_HOOK), used to model
// lock-step chains and placements (DESIGN.md section 5).  g++ -O2 -fopenmp -shared -fPIC -x c++ -Iinclude -o build/libsteps_quad_day.so scripts/steps_quad_day.cpp
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#define SP_DAY_HOOK(io, day, n) (io).hook(day, n)
#include "../simplyp_b200/csrc/simplyp_quad.cuh"
using namespace simplyp;
struct IO {
  const double* f; const ThreadCounters* cnt; uint16_t* steps; long long last;
  void wait(int) const {}
  void forcing(int day, double& P, double& E, double& doy, double& T) const { P = f[4*day]; E = f[4*day+1]; doy = f[4*day+2]; T = f[4*day+3]; }
  void upstream(int, double (&us)[4]) const { us[0]=us[1]=us[2]=us[3]=0; }
  bool wants_vr() const { return false; }
  void publish(int) const {}
  void hook(int day, unsigned n) { steps[day] = (uint16_t)(n - last); last = n; }
  template <class Q> void emit(const Q&, int day, const double (&)[NL], double, const double (&acc)[NA], const double (&)[13], const Cold&) {}
};
extern "C" int steps_quad_day(int M, int D, const double* forcing, const double* mp, const double* scp, double rtol, double atol, uint16_t* steps) {
  ThreadOptions t; memset(&t, 0, sizeof(t)); t.rtol = rtol; t.atol = atol; t.step_len = 1.0; t.max_steps_per_day = 5000;
  t.dynamic_epc0 = 1; t.dynamic_erod = 1; t.run_mode_cal = 1; t.strict_quirks = 1;
#pragma omp parallel for schedule(dynamic, 16)
  for (int m = 0; m < M; ++m) {
    ThreadCounters cnt; QuadMem qm; QuadHost4 q; IO io{forcing, &cnt, steps + (size_t)m * D, 0};
    run_quad<false>(q, mp + (size_t)m * SIMPLYP_NP_MEMBER, scp, scp[SIMPLYP_SC_A_CATCH], 0, t, D, true, qm, io, cnt);
  }
  return 0;
}
