// Analysis tool: every step attempt of the quad program on the host (SP_ATTEMPT_HOOK): where in the day the attempts and
// the rejections fall, and how the first step of a day compares with the step the controller would have liked.
//   g++ -O2 -fopenmp -std=c++17 -shared -fPIC -o build/libsteps_attempts.so scripts/steps_attempts.cpp
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#define SP_ATTEMPT_HOOK(io, day, k, t, hh, en2, acc) (io).hook(day, k, t, hh, en2, acc)
#include "../simplyp_b200/csrc/simplyp_quad.cuh"
using namespace simplyp;
struct Rec { float t, h, en2; int16_t k; int8_t acc; int8_t pad; };
struct IO {
  const double* f; Rec* rec; int* nrec; int D; int cap;
  void wait(int) const {}
  void forcing(int day, double& P, double& E, double& doy, double& T) const { P = f[4*day]; E = f[4*day+1]; doy = f[4*day+2]; T = f[4*day+3]; }
  void upstream(int, double (&us)[4]) const { us[0]=us[1]=us[2]=us[3]=0; }
  void publish(int) const {}
  void hook(int day, int k, double t, double hh, double en2, bool acc) {
    // first 6 attempts of each day + the last
    if (k <= cap) { Rec& r = rec[(size_t)day * cap + (k - 1)]; r.t = (float)t; r.h = (float)hh; r.en2 = (float)en2; r.k = (int16_t)k; r.acc = acc; }
    nrec[day] = k;
  }
  template <class Q> void emit(const Q&, int, const double (&)[NL], double, const double (&)[NA], const double (&)[13], const Cold&) {}
};
extern "C" int steps_attempts(int M, int D, int cap, const double* forcing, const double* mp, const double* scp, double rtol, double atol,
                              Rec* rec, int* nrec) {
  ThreadOptions t; memset(&t, 0, sizeof(t)); t.rtol = rtol; t.atol = atol; t.step_len = 1.0; t.max_steps_per_day = 5000;
  t.dynamic_epc0 = 1; t.dynamic_erod = 1; t.run_mode_cal = 1; t.strict_quirks = 1;
#pragma omp parallel for schedule(dynamic, 16)
  for (int m = 0; m < M; ++m) {
    ThreadCounters cnt; QuadMem qm; QuadHost4 q; IO io{forcing, rec + (size_t)m * D * cap, nrec + (size_t)m * D, D, cap};
    run_quad<false>(q, mp + (size_t)m * SIMPLYP_NP_MEMBER, scp, scp[SIMPLYP_SC_A_CATCH], 0, t, D, true, qm, io, cnt);
  }
  return 0;
}
