// simplyp_quad.cuh — one (ensemble member, sub-catchment) integrated by a QUAD of 4 adjacent lanes.
//
// Why: with one thread per member a 10^4-member ensemble is 313 warps on 592 SM sub-partitions and every
// thread is one long dependent fp64 chain (measured 3.3 cycles per issued instruction, 8.1-cycle DFMA
// latency): the run is latency-bound and most of the machine idles.  ode_f (model.py:58-187) however has
// four-fold structure: two identical soil boxes, a groundwater box and a reach whose in-stream masses obey
// the same linear equation.  The 12 ODE components of ode_f are dealt to 4 lanes, 3 each:
//
//      lane   slot A        slot B     accumulator     own exponential        own gate (f_x)
//      0      VsA   y[0]    Msus y[6]  Msus_out y[7]   exp(-mu VsA)           soil A       -> QsA
//      1      VsS   y[1]    TDPr y[8]  TDPr_out y[9]   exp(-mu VsS)           soil S       -> QsS
//      2      Vg    y[2]    PPr  y[10] PPr_out  y[11]  Qr^k_M = exp(k_M u)    groundwater  -> Qg
//      3      u=ln Qr y[4]  Vr   y[3]  Qr_av    y[5]   Qr    = exp(u)         (none)
//
// Every lane executes the SAME instruction stream on lane-specific coefficients (QuadCoef), so there is no
// divergence inside a quad: ONE exp and ONE gate per lane per RHS evaluation (the scalar program issues
// log + 4 exp + 3 gates per thread), seven 64-bit quad broadcasts, two short linear forms.
//   * Qr is carried as u = ln Qr:  dQr/dt = net*a_Q*Qr^b_Q*86400/((1-b_Q) L)  (:127-130)  becomes
//     du/dt = net / ((1-b_Q) Vr)  because ode_f's dVr/dt = net (:131) and the initial condition (:457-459)
//     keep Vr = L/(a_Q 86400) Qr^(1-b_Q).  No logarithm and no Qr^b_Q are needed: Qr/Vr (the outflow rate of
//     Msus, TDPr, PPr, :145-180) is exp(u) * rcp(Vr).  Vr is integrated, as in the reference.
//   * The error norm is LSODA's: scaled RMS over all 12 components (u is weighted so that its term equals
//     the one Qr would have had: err_u * Qr / (atol + rtol*Qr)).
// The once-a-day algebra (begin_day / end_day of simplyp_core.cuh) is executed redundantly by the 4 lanes
// on values gathered with quad broadcasts; results are identical on the 4 lanes by construction.
//
// A warp holds 8 quads and advances them through the days in LOCK-STEP: the step loop of a day runs until
// the slowest quad has reached midnight (finished quads execute the attempt without committing it), so the
// day-boundary code is executed once per warp-day and the control flow of a warp is uniform.  Measured on
// the bench ensemble (scripts/policy_analysis.py): lane efficiency 0.73 unsorted / 0.875 with members ordered
// by a short pilot run, against 0.70 for 32 independent members per warp in a flattened loop.
//
// The program is written once, generic in an execution policy Q:
//   QuadDev   (device): T = double, quad broadcasts are __shfl_sync(..., width 4)
//   QuadHost4 (tests/hostemu only): T = V4, the 4 lanes are the 4 elements of a struct
#pragma once

#include "simplyp_core.cuh"

#ifndef SP_DAYSTART_FAC
#define SP_DAYSTART_FAC 0.2   // day-start step = this x yesterday's last step (the forcing jumps at midnight);
                              // 0.1 / 0.3 / 0.5 and "yesterday's first accepted step" all need more attempts
                              // (scripts/controller_exp.py)
#endif
#ifndef SP_TOL_RATE0
#define SP_TOL_RATE0 5.0      // reach rate constant (per day) above which the day's tolerance grows with the rate ...
#define SP_TOL_GMAX 8.0       // ... up to this factor (see run_quad)
#endif
#ifndef SP_STIFF_RATE
#define SP_STIFF_RATE 80.0    // reach rate constant Qr/((1-b_Q) Vr) per day above which a day is integrated by the
                              // Rosenbrock path: the explicit pair is stability-bound there (~rate/3.3 attempts per
                              // day), the Rosenbrock path needs 25-40 whatever the rate since its error norm relaxes
                              // the reach's own terms (SP_ROS_RATE0); round 1 switched at 150 per day (45-55 attempts)
#endif
#ifndef SP_ROS_TOL_SCALE
#define SP_ROS_TOL_SCALE 30.0 // Kaps-Rentrop's 3rd-order estimate is conservative: at 30x the tolerance the flows of a
                              // stiff reach are still within 5e-7 of LSODA/BDF at 1e-10 and its end-of-day states
                              // within 3e-6 (tests/...::test_stiff_reach_*), the explicit pair's own level
#endif
#ifndef SP_ROS_RATE0
#define SP_ROS_RATE0 80.0     // Rosenbrock days: the error terms of the reach and of what it carries (u, Vr, in-stream masses,
#define SP_ROS_GMAX 30.0      // daily sums) are relaxed by rate/SP_ROS_RATE0, at most SP_ROS_GMAX-fold, except in the last
#endif                        // step of the day (the end-of-day states are outputs); see run_quad
#ifndef SP_ROS_W_SOIL
#define SP_ROS_W_SOIL 3.0     // ... while the soil volumes and the groundwater are held 3x tighter than the Rosenbrock
#define SP_ROS_W_VG 3.0       // tolerance scale alone would (a stiff reach does not make its land phase stiff)
#endif
#ifndef SP_H0_STIFF_C
#define SP_H0_STIFF_C 0.15    // first step of a Rosenbrock day <= this / rate: the boundary layer the midnight jump of the
#endif                        // forcing excites is ~1/rate wide (saves the 5-6 rejections that found this step size)
// Analysis knobs of the explicit pair's error norm (scripts/errnorm_exp.py, errnorm_validate.py); at 1.0 — the product's
// setting: lower weights cost more accuracy on the light members than they save attempts, DESIGN.md section 4 — the
// multiplications fold away.
#ifndef SP_W_B
#define SP_W_B 1.0     // weight of the slot-B (in-stream masses, Vr) terms of the error norm
#define SP_W_ACC 1.0   // weight of the daily accumulators
#endif
#ifndef SP_W_U
#define SP_W_U 1.0     // weight of the u = ln Qr term of the error norm
#endif
#ifndef SP_W_VG
#define SP_W_VG 1.0    // weight of the groundwater volume
#endif
#ifndef SP_SOIL_ERR_WEIGHT
#define SP_SOIL_ERR_WEIGHT 1000.0
#endif

namespace simplyp {

// ------------------------------------------------------------------------------------------ section probe
// Analysis builds (-DSP_LAT_PROBE, scripts/exp_lat_sections.py): every warp reads clock64() at the section boundaries of
// its day loop and adds the cycles between two reads to the section the second one closes.  A boundary is where the
// read ISSUES: a result still in flight there is charged to the section that waits for it.  Without the macro the
// marks are empty and the product build is unchanged.
#if defined(SP_LAT_PROBE) && defined(__CUDA_ARCH__)
enum { LP_RHS = 0,   // step loop top -> the attempt's sixth RHS evaluation (stage arguments included)
       LP_ERR,       // -> the error norm en2
       LP_CTRL,      // -> the end of the loop body: controller, accept/reject bookkeeping
       LP_END,       // step loop exit (last vote) -> end of the day: state gather, end_day, statistics, barriers
       LP_START,     // -> entry of tomorrow's step loop: wait / forcing, begin_day, quad_daily_coef, first RHS + Jacobian
       LP_ITERS,     // step-loop iterations of the warp (attempts in lock-step)
       LP_DAYS,      // day boundaries
       LP_N };
static_assert(LP_N <= 8, "ThreadCounters::lat");
struct LatProbe {
  long long t, acc[LP_N];
  __device__ __forceinline__ void mark(int sec) { const long long c = clock64(); acc[sec] += c - t; t = c; }
};
#define SP_LAT_PARAM , LatProbe& lp
#define SP_LAT_ARG , lp
#define SP_LAT_MARK(sec) lp.mark(sec)
#define SP_LAT_COUNT(i) (++lp.acc[i])
#else
#define SP_LAT_PARAM
#define SP_LAT_ARG
#define SP_LAT_MARK(sec) ((void)0)
#define SP_LAT_COUNT(i) ((void)0)
#endif

// ------------------------------------------------------------------------------------------ 4-lane host value
struct V4 { double v[4]; };
#define SP_V4_BIN(op)                                                                                             \
  inline V4 operator op(const V4& a, const V4& b) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = a.v[l] op b.v[l]; return r; } \
  inline V4 operator op(const V4& a, double b) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = a.v[l] op b; return r; }         \
  inline V4 operator op(double a, const V4& b) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = a op b.v[l]; return r; }
SP_V4_BIN(+) SP_V4_BIN(-) SP_V4_BIN(*)
#undef SP_V4_BIN
inline V4 v4_splat(double x) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = x; return r; }

// elementary operations on T (double on the device, V4 in the host harness)
SP_HD double qfma(double a, double b, double c) { return fma(a, b, c); }
SP_HD double qgate(double u) { return gate(u); }
SP_HD double qclamp01(double u) { return sp_clamp01(u); }
SP_HD double qrcp(double x) { return sp_rcp(x); }
SP_HD double qrcp40(double x) { return sp_rcp40(x); }
SP_HD double qrcp_fast(double x) { return sp_rcp_fast(x); }
SP_HD double qabs(double x) { return fabs(x); }
SP_HD double qmax(double a, double b) { return sp_max(a, b); }
#define SP_V4_MAP1(name, f) inline V4 name(const V4& a) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = f(a.v[l]); return r; }
SP_V4_MAP1(qgate, gate) SP_V4_MAP1(qclamp01, sp_clamp01) SP_V4_MAP1(qrcp, sp_rcp) SP_V4_MAP1(qrcp40, sp_rcp40) SP_V4_MAP1(qrcp_fast, sp_rcp_fast)
SP_V4_MAP1(qabs, fabs)
#undef SP_V4_MAP1
inline V4 qmax(const V4& a, const V4& b) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = sp_max(a.v[l], b.v[l]); return r; }
inline V4 qfma(const V4& a, const V4& b, const V4& c) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = fma(a.v[l], b.v[l], c.v[l]); return r; }
inline V4 qfma(double a, const V4& b, const V4& c) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = fma(a, b.v[l], c.v[l]); return r; }
inline V4 qfma(const V4& a, double b, const V4& c) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = fma(a.v[l], b, c.v[l]); return r; }
inline V4 qfma(const V4& a, const V4& b, double c) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = fma(a.v[l], b.v[l], c); return r; }
inline V4 qfma(double a, const V4& b, double c) { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = fma(a, b.v[l], c); return r; }

// ------------------------------------------------------------------------------------------ execution policies
struct QuadHost4 {
  using T = V4;
  T pick(double a, double b, double c, double d) const { return V4{{a, b, c, d}}; }
  T splat(double x) const { return v4_splat(x); }
  T exp(const T& x) const { V4 r; for (int l = 0; l < 4; ++l) r.v[l] = sp_exp_tab(x.v[l], kExp2Tab); return r; }
  T bcast(const T& x, int src) const { return v4_splat(x.v[src]); }
  T sum(const T& x) const { return v4_splat((x.v[0] + x.v[1]) + (x.v[2] + x.v[3])); }   // butterfly order
  double first(const T& x) const { return x.v[0]; }                                  // quad-uniform values only
  T sel3(const T& on3, const T& other) const { return V4{{other.v[0], other.v[1], other.v[2], on3.v[3]}}; }
  bool any(bool p) const { return p; }
  bool leader() const { return true; }
  void sync() const {}
};

#if defined(__CUDACC__)
struct QuadDev {
  using T = double;
  int ql;              // lane within the quad
  const double* tab;   // 2^(j/32) table in shared memory
  __device__ __forceinline__ T exp(T x) const { return sp_exp_tab(x, tab); }
  __device__ __forceinline__ T pick(double a, double b, double c, double d) const {
    return ql == 0 ? a : (ql == 1 ? b : (ql == 2 ? c : d));
  }
  __device__ __forceinline__ T splat(double x) const { return x; }
  __device__ __forceinline__ T bcast(T x, int src) const {
    // the two halves are shuffled as ints: __shfl_sync(double) makes ptxas swap the register pair afterwards
#ifdef SP_BCAST_DOUBLE
    return __shfl_sync(0xffffffffu, x, src, 4);
#else
    const int lo = __shfl_sync(0xffffffffu, __double2loint(x), src, 4);
    const int hi = __shfl_sync(0xffffffffu, __double2hiint(x), src, 4);
    return __hiloint2double(hi, lo);
#endif
  }
  // (x + x^1) + (x^2 + x^3): the butterfly's value on every lane (fp addition commutes bitwise, so lane 2's
  // (x2 + x3) + (x0 + x1) is lane 0's sum), but the three fetches are independent — one shuffle round trip on the
  // error norm's dependent path instead of two
  __device__ __forceinline__ T sum(T x) const {
    const T x1 = __shfl_xor_sync(0xffffffffu, x, 1);
    const T x2 = __shfl_xor_sync(0xffffffffu, x, 2);
    const T x3 = __shfl_xor_sync(0xffffffffu, x, 3);
    return (x + x1) + (x2 + x3);
  }
  __device__ __forceinline__ double first(T x) const { return x; }
  __device__ __forceinline__ T sel3(T on3, T other) const { return ql == 3 ? on3 : other; }
  __device__ __forceinline__ bool any(bool p) const { return __any_sync(0xffffffffu, p) != 0; }
  __device__ __forceinline__ bool leader() const { return ql == 0; }
  __device__ __forceinline__ void sync() const { __syncwarp(); }
};
#endif

// ------------------------------------------------------------------------------------------ lane coefficients
template <class Q>
struct QuadCoef {
  using T = typename Q::T;
  T eY, eU;                    // own exponential: exp(eY*yA + eU*u)
  T p1, p0, g0, g1;            // own gate: w = p1*yA + p0 ; G = g0 + f(w)*w*g1   (f = smoothstep on [0,1])
  T a0, aE, aSA, aSS, aG, aR;  // slot A: L = a0 + aE*e + aSA*QsA + aSS*QsS + aG*Qg + aR*Qr ; dA = L*(m0 + mA/Vr)
  T aRE;                       //   aE (lanes 0-2) and aR (lane 3) in one coefficient of the own exponential: lane 3's
                               //   own exponential IS Qr, and its aE is zero like the other lanes' aR
  T m0, mA;                    //   lanes 0-2: (1, 0) ; lane 3: (0, 1/(1-b_Q))  -> du/dt = net/((1-b_Q) Vr)
  T rvOff;                     //   added to slot B before the reciprocal: 0 on lane 3 (1/Vr), 1 elsewhere (the other
                               //   lanes' mA is zero; the offset only keeps their unused reciprocal finite)
  T b0, bK, bSA, bSS, bG;      // slot B: dB = b0 + bK*Qr^k + bSA*QsA + bSS*QsS + bG*Qg - yB*Qr/Vr
};                             //   lane 3 (yB = Vr): yB*Qr/Vr = Qr, so its b-coefficients spell net + Qr (:127,131)

// Coefficients that do not change from day to day (member constants), from the scalar program's Hot.
template <class Q>
SP_HD void quad_static_coef(const Q& q, const Hot& h, QuadCoef<Q>& c) {
  const double omb = 1.0 - h.beta;
  c.eY = q.pick(-h.mu, -h.mu, 0.0, 1.0);
  c.eU = q.pick(0.0, 0.0, h.kM, 0.0);
  // soil boxes (:105,109): w = (Vs-fc)/(0.01 fc), Qs = (Vs-fc) f(w)/T_s = w f(w) (0.01 fc/T_s)
  // groundwater (:121-122): w = (Vg/T_g-Qg_min)/(0.01 Qg_min), Qg = Qg_min + f(w) w (0.01 Qg_min)
  const double fcd = h.fc * 0.01, qgd = h.Qg_min * 0.01;
  c.p1 = q.pick(h.inv_fcd, h.inv_fcd, h.inv_Tg * h.inv_Qgd, 0.0);
  c.p0 = q.pick(-h.fc * h.inv_fcd, -h.fc * h.inv_fcd, -h.Qg_min * h.inv_Qgd, 0.0);
  c.g0 = q.pick(0.0, 0.0, h.Qg_min, 0.0);
  c.g1 = q.pick(fcd * h.inv_TsA, fcd * h.inv_TsS, qgd, 0.0);
  c.aSA = q.pick(-1.0, 0.0, h.beta * h.fA, omb * h.fA);          // :106, :124, :127
  c.aSS = q.pick(0.0, -1.0, h.beta * h.fS, omb * h.fS);
  c.aG = q.pick(0.0, 0.0, -1.0, 1.0);
  c.aR = q.pick(0.0, 0.0, 0.0, -1.0);
  c.m0 = q.pick(1.0, 1.0, 1.0, 0.0);
  c.mA = q.pick(0.0, 0.0, 0.0, 1.0 / (1.0 - h.bQ));
  c.rvOff = q.pick(1.0, 1.0, 1.0, 0.0);
  c.bG = q.pick(0.0, h.tG, 0.0, 1.0);                            // :163 ; lane 3: +Qg
  c.a0 = c.aE = c.aRE = c.b0 = c.bK = c.bSA = c.bSS = q.splat(0.0);
}

// Coefficients that follow the day's forcing, upstream inputs and soil-P carry (filled by begin_day in h).
template <class Q>
SP_HD void quad_daily_coef(const Q& q, const Hot& h, QuadCoef<Q>& c) {
  c.a0 = q.pick(h.Pin - h.aE, h.Pin - h.aE, 0.0, h.qin0);        // :106,110 ; :127
  c.aE = q.pick(h.aE, h.aE, 0.0, 0.0);
  c.aRE = q.pick(h.aE, h.aE, 0.0, -1.0);
  const double omb = 1.0 - h.beta;
  c.b0 = q.pick(h.MsusUS, h.t0, h.PPUS, h.qin0);                 // :144, :165-166, :177 ; lane 3: :127
  c.bK = q.pick(h.cM, 0.0, h.cP, 0.0);                           // :138-143, :171-176
  c.bSA = q.pick(0.0, h.tA, 0.0, omb * h.fA);                    // :154-161
  c.bSS = q.pick(0.0, h.tS, 0.0, omb * h.fS);
}

// One evaluation of ode_f by the quad.  `e` returns the lane's own exponential (lane 3: Qr at this state).
template <class Q>
SP_HD void quad_rhs(const Q& q, const QuadCoef<Q>& c, const typename Q::T& yA, const typename Q::T& yB,
                    typename Q::T& dA, typename Q::T& dB, typename Q::T& dacc, typename Q::T& e) {
  using T = typename Q::T;
  // Source order = intended issue order (ptxas keeps independent chains roughly where they are written): the gated
  // flows depend on the lane's own state only, so they are computed and broadcast FIRST; the exponential, which
  // waits for the broadcast of u, then has only its own two broadcasts behind it.
  // Six quad broadcasts: u, the three gated flows, Qr^k_M and the outflow rate Qr/Vr.  Lane 3 owns both Qr (its
  // exponential) and Vr (its slot B), so it forms Qr/Vr itself and nobody else needs Vr or Qr.
  const T w = qfma(c.p1, yA, c.p0);
  const T G = qfma(qgate(w) * w, c.g1, c.g0);
  const T u = q.bcast(yA, 3);
  const T rV = qrcp40(yB + c.rvOff);        // lane 3: 1/Vr to 40 bits (the integration tolerance is 1e-7)
  const T QsA = q.bcast(G, 0), QsS = q.bcast(G, 1), Qg = q.bcast(G, 2);
  e = q.exp(qfma(c.eU, u, c.eY * yA));      // (the product that does not wait for the broadcast is formed first)
  const T gsum = qfma(c.aG, Qg, qfma(c.aSA, QsA, qfma(c.aSS, QsS, c.a0)));   // ready before the exponential
  const T src0 = qfma(c.bSA, QsA, qfma(c.bSS, QsS, qfma(c.bG, Qg, c.b0)));
  const T mult = qfma(rV, c.mA, c.m0);
  const T qk = q.bcast(e, 2);
  const T r = q.bcast(e * rV, 3);           // Qr/Vr
  const T L = qfma(c.aRE, e, gsum);
  const T out = yB * r;                      // outflow of the lane's in-stream mass (:145,147,166,168,178,180)
  dA = L * mult;                             // lane 3: du/dt = net/((1-b_Q) Vr)
  dB = qfma(c.bK, qk, src0) - out;           // lane 3: out = Vr*Qr/Vr = Qr, src = net + Qr -> dVr/dt = net (:131)
  dacc = out;                                // lane 3: dQr_av/dt = Qr (:132)
}

// Per-lane Runge-Kutta state.
template <class Q>
struct QuadState {
  using T = typename Q::T;
  T yA, yB, acc;        // the lane's three components
  T k1A, k1B, a1;       // derivatives at the current point (FSAL / reused after a rejection)
  T e1;                 // own exponential at the current point (lane 3: Qr)
};

// One embedded RK5(4) step attempt of the quad.  Returns the MEAN SQUARE of the scaled error over the 12
// components (same on all lanes); <= 1 accepts.
template <class Q>
SP_HD double quad_attempt(const Q& q, const QuadCoef<Q>& c, const QuadState<Q>& s, double hh, double rtol, double atol,
                          typename Q::T& ynA, typename Q::T& ynB, typename Q::T& accn, typename Q::T& k7A,
                          typename Q::T& k7B, typename Q::T& a7, typename Q::T& e7o SP_LAT_PARAM) {
  using T = typename Q::T;
  T kA2, kA3, kA4, kA5, kA6, kB2, kB3, kB4, kB5, kB6, da, ee;
  T sb = kRK[RB1] * s.a1, se = kRK[RE1] * s.a1;
  quad_rhs(q, c, qfma(hh, kRK[RA21] * s.k1A, s.yA), qfma(hh, kRK[RA21] * s.k1B, s.yB), kA2, kB2, da, ee);
  sb = qfma(kRK[RB2], da, sb); se = qfma(kRK[RE2], da, se);
  quad_rhs(q, c, qfma(hh, qfma(kRK[RA32], kA2, kRK[RA31] * s.k1A), s.yA), qfma(hh, qfma(kRK[RA32], kB2, kRK[RA31] * s.k1B), s.yB), kA3, kB3, da, ee);
  sb = qfma(kRK[RB3], da, sb); se = qfma(kRK[RE3], da, se);
  quad_rhs(q, c, qfma(hh, qfma(kRK[RA43], kA3, qfma(kRK[RA42], kA2, kRK[RA41] * s.k1A)), s.yA),
           qfma(hh, qfma(kRK[RA43], kB3, qfma(kRK[RA42], kB2, kRK[RA41] * s.k1B)), s.yB), kA4, kB4, da, ee);
  sb = qfma(kRK[RB4], da, sb); se = qfma(kRK[RE4], da, se);
  quad_rhs(q, c, qfma(hh, qfma(kRK[RA54], kA4, qfma(kRK[RA53], kA3, qfma(kRK[RA52], kA2, kRK[RA51] * s.k1A))), s.yA),
           qfma(hh, qfma(kRK[RA54], kB4, qfma(kRK[RA53], kB3, qfma(kRK[RA52], kB2, kRK[RA51] * s.k1B))), s.yB), kA5, kB5, da, ee);
  sb = qfma(kRK[RB5], da, sb); se = qfma(kRK[RE5], da, se);
  quad_rhs(q, c, qfma(hh, qfma(kRK[RA65], kA5, qfma(kRK[RA64], kA4, qfma(kRK[RA63], kA3, qfma(kRK[RA62], kA2, kRK[RA61] * s.k1A)))), s.yA),
           qfma(hh, qfma(kRK[RA65], kB5, qfma(kRK[RA64], kB4, qfma(kRK[RA63], kB3, qfma(kRK[RA62], kB2, kRK[RA61] * s.k1B)))), s.yB), kA6, kB6, da, ee);
  sb = qfma(kRK[RB6], da, sb); se = qfma(kRK[RE6], da, se);
  ynA = qfma(hh, qfma(kRK[RB6], kA6, qfma(kRK[RB5], kA5, qfma(kRK[RB4], kA4, qfma(kRK[RB3], kA3, qfma(kRK[RB2], kA2, kRK[RB1] * s.k1A))))), s.yA);
  ynB = qfma(hh, qfma(kRK[RB6], kB6, qfma(kRK[RB5], kB5, qfma(kRK[RB4], kB4, qfma(kRK[RB3], kB3, qfma(kRK[RB2], kB2, kRK[RB1] * s.k1B))))), s.yB);
  quad_rhs(q, c, ynA, ynB, k7A, k7B, a7, e7o);
  SP_LAT_MARK(LP_RHS);
  accn = qfma(hh, sb, s.acc);
  const T eA = hh * qfma(kRK[RE7], k7A, qfma(kRK[RE6], kA6, qfma(kRK[RE5], kA5, qfma(kRK[RE4], kA4, qfma(kRK[RE3], kA3, qfma(kRK[RE2], kA2, kRK[RE1] * s.k1A))))));
  const T eB = hh * qfma(kRK[RE7], k7B, qfma(kRK[RE6], kB6, qfma(kRK[RE5], kB5, qfma(kRK[RE4], kB4, qfma(kRK[RE3], kB3, qfma(kRK[RE2], kB2, kRK[RE1] * s.k1B))))));
  const T ec = hh * qfma(kRK[RE7], a7, se);
  // error weights (odeint: atol + rtol*|y|).  Lane 3's slot A is u = ln Qr: err_Qr = Qr err_u, scale on Qr.
  const T Qmax = qmax(s.e1, e7o);
  const T sA = q.sel3(Qmax, qmax(qabs(s.yA), qabs(ynA)));
  const T wA = q.sel3(Qmax * SP_W_U, q.pick(SP_SOIL_ERR_WEIGHT, SP_SOIL_ERR_WEIGHT, SP_W_VG, 1.0));
  const T qA = (eA * wA) * qrcp_fast(qfma(rtol, sA, atol));
  const T qB = (eB * SP_W_B) * qrcp_fast(qfma(rtol, qmax(qabs(s.yB), qabs(ynB)), atol));
  const T qc = (ec * SP_W_ACC) * qrcp_fast(qfma(rtol, qmax(qabs(s.acc), qabs(accn)), atol));
  // (a NaN is returned as it is: it rejects like +inf, and step_factor_sq gives both the smallest factor — no select
  // on the controller's dependent path)
  return q.first(q.sum(qfma(qA, qA, qfma(qB, qB, qc * qc)))) * (1.0 / 12.0);
}

// ------------------------------------------------------------------------------------------ stiff reaches
// In a large network a main-stem reach carries the runoff of thousands of km2 over its own small area; its rate
// constant Qr/((1-b_Q) Vr) then reaches 1e3 per day and the explicit pair becomes stability-bound (hundreds of
// attempts per day).  LSODA switches to BDF there (model.py:640); this path switches, per item and per day, to a
// linearly-implicit (Rosenbrock) method: Kaps-Rentrop 4(3) with Shampine's parameters (4 stages, 3 RHS
// evaluations, L-stable-ish, embedded 3rd-order error estimate), with the EXACT Jacobian of ode_f.
// The Jacobian is block lower-triangular in the order (VsA, VsS) -> Vg -> (u, Vr) -> (Msus, TDPr, PPr) -> the four
// quadratures, so (I/(gamma h) - J) g = rhs is solved by forward substitution: lanes 0 and 1 divide, lane 2 divides
// after receiving their results, lane 3 solves a 2x2 system, lanes 0-2 then finish their in-stream mass and every
// lane its quadrature — five quad broadcasts per solve, no pivoting, no matrix in memory.
namespace ros {
constexpr double GAM = 0.5;
constexpr double A21 = 2.0, A31 = 48.0 / 25.0, A32 = 6.0 / 25.0;
constexpr double C21 = -8.0, C31 = 372.0 / 25.0, C32 = 12.0 / 5.0, C41 = -112.0 / 125.0, C42 = -54.0 / 125.0, C43 = -2.0 / 5.0;
constexpr double B1 = 19.0 / 9.0, B2 = 0.5, B3 = 25.0 / 108.0, B4 = 125.0 / 108.0;
constexpr double E1 = 17.0 / 54.0, E2 = 7.0 / 36.0, E3 = 0.0, E4 = 125.0 / 108.0;
}  // namespace ros

// Lane-local entries of the Jacobian of ode_f at one state (d = derivative of the row's component).
template <class Q>
struct QuadJac {
  using T = typename Q::T;
  T dAA;                  // slot A diagonal (lane 3: d(du)/du)
  T jA1, jA2, jA3;        // slot A row: d/dVsA, d/dVsS, d/dVg   (zero where the column is the row itself or later)
  T jB1, jB2, jB3;        // slot B row: d/dVsA, d/dVsS, d/dVg
  T jB4, jB5, dBB;        // slot B row: d/du, d/dVr, diagonal   (lane 3 = Vr row: jB4 = -Qr, jB5 = dBB = 0)
  T jC1, jC2, jC3;        // accumulator row: d/d(own slot B), d/du, d/dVr
  T jUV;                  // lane 3: d(du)/dVr
};

// ode_f and its Jacobian at (yA, yB): returns the derivatives like quad_rhs and fills J.
template <class Q>
SP_HD void quad_rhs_jac(const Q& q, const QuadCoef<Q>& c, const typename Q::T& yA, const typename Q::T& yB,
                        typename Q::T& dA, typename Q::T& dB, typename Q::T& dacc, typename Q::T& e, QuadJac<Q>& J) {
  using T = typename Q::T;
  const T u = q.bcast(yA, 3);
  const T rV = qrcp(q.bcast(yB, 3));
  e = q.exp(qfma(c.eY, yA, c.eU * u));
  const T w = qfma(c.p1, yA, c.p0);
  const T wc = qclamp01(w);
  const T fw = wc * wc * (3.0 - 2.0 * wc);
  const T G = qfma(fw * w, c.g1, c.g0);
  const T dG = (c.g1 * c.p1) * qfma(w * 6.0, wc * (1.0 - wc), fw);          // dG/d(own slot A)
  const T QsA = q.bcast(G, 0), QsS = q.bcast(G, 1), Qg = q.bcast(G, 2);
  const T dGA = q.bcast(dG, 0), dGS = q.bcast(dG, 1), dGg = q.bcast(dG, 2);
  const T qk = q.bcast(e, 2), Qr = q.bcast(e, 3);
  const T L = (qfma(c.aE, e, c.a0) + qfma(c.aSA, QsA, c.aSS * QsS)) + qfma(c.aG, Qg, c.aR * Qr);
  const T r = Qr * rV;
  const T out = yB * r;
  const T src = qfma(c.bK, qk, c.b0) + qfma(c.bSA, QsA, qfma(c.bSS, QsS, c.bG * Qg));
  const T mult = qfma(rV, c.mA, c.m0);
  dA = L * mult;
  dB = src - out;
  dacc = out;
  // slot A: lanes 0,1 depend on themselves only; lane 2 (Vg) on VsA, VsS, itself; lane 3 (u) on all of them, u, Vr
  const T up = q.pick(0.0, 0.0, 1.0, 1.0), up3 = q.pick(0.0, 0.0, 0.0, 1.0);
  const T own = q.pick(-1.0, -1.0, -1.0, 0.0);                                 // coefficient of the own gated flow
  J.dAA = (qfma(c.aE * c.eY, e, own * dG) + c.aR * Qr) * mult;
  J.jA1 = up * c.aSA * dGA * mult;
  J.jA2 = up * c.aSS * dGS * mult;
  J.jA3 = up3 * c.aG * dGg * mult;
  J.jUV = (0.0 - dA) * rV;                                                     // lane 3: d(net m)/dVr, m = mA/Vr
  // slot B: in-stream masses (lanes 0-2), Vr (lane 3)
  J.jB1 = c.bSA * dGA;
  J.jB2 = c.bSS * dGS;
  J.jB3 = c.bG * dGg;
  J.jB4 = qfma(c.bK * q.bcast(c.eU, 2), qk, 0.0 - out);                        // d/du: k_M bK Qr^k_M - yB r (lane 3: -Qr)
  J.jB5 = q.sel3(q.splat(0.0), out * rV);                                      // d/dVr: yB r / Vr
  J.dBB = q.sel3(q.splat(0.0), 0.0 - r);
  // accumulators: d(yB r) (lane 3: dQr = Qr du)
  J.jC1 = q.sel3(q.splat(0.0), r);
  J.jC2 = out;
  J.jC3 = q.sel3(q.splat(0.0), (0.0 - out) * rV);
}

// Factors of (I/(gamma h) - J) that depend on the step size.
template <class Q>
struct QuadLU {
  using T = typename Q::T;
  T m11, m12, m21, m22;   // lanes 0-2: m11 = 1/(d - dAA), others 0; lane 3: inverse of the (u, Vr) 2x2 block
  T idB;                  // lanes 0-2: 1/(d - dBB)
  double gh;              // gamma h = 1/d
};

template <class Q>
SP_HD void quad_factor(const Q& q, const QuadJac<Q>& J, double hh, QuadLU<Q>& F) {
  using T = typename Q::T;
  const double d = sp_rcp(ros::GAM * hh);      // (sp_rcp, not '/': no division subroutine in the step loop)
  F.gh = ros::GAM * hh;
  const T a = d - J.dAA;
  // lane 3: [a, -jUV; -jB4, d]^-1 = 1/det [d, jUV; jB4, a]
  const T det = q.sel3(a * d - J.jUV * J.jB4, a);
  const T idet = qrcp(det);
  F.m11 = q.sel3(d * idet, idet);
  F.m12 = q.sel3(J.jUV * idet, q.splat(0.0));
  F.m21 = q.sel3(J.jB4 * idet, q.splat(0.0));
  F.m22 = q.sel3(a * idet, q.splat(0.0));
  F.idB = qrcp(d - J.dBB);
}

// g = (I/(gamma h) - J)^-1 rhs for the lane's three components.
template <class Q>
SP_HD void quad_solve(const Q& q, const QuadJac<Q>& J, const QuadLU<Q>& F, const typename Q::T& rA, const typename Q::T& rB,
                      const typename Q::T& rC, typename Q::T& gA, typename Q::T& gB, typename Q::T& gC) {
  using T = typename Q::T;
  const T g0 = rA * F.m11;                                   // final on lanes 0,1
  const T gVsA = q.bcast(g0, 0), gVsS = q.bcast(g0, 1);
  T t1 = qfma(J.jA1, gVsA, qfma(J.jA2, gVsS, rA));
  T t2 = qfma(J.jB1, gVsA, qfma(J.jB2, gVsS, rB));
  const T gVg = q.bcast(t1 * F.m11, 2);                      // final on lane 2
  t1 = qfma(J.jA3, gVg, t1);
  t2 = qfma(J.jB3, gVg, t2);
  gA = qfma(F.m11, t1, F.m12 * t2);                          // lane 3: g_u ; lanes 0-2: their slot A
  const T y = qfma(F.m21, t1, F.m22 * t2);                   // lane 3: g_Vr
  const T gu = q.bcast(gA, 3), gV = q.bcast(y, 3);
  gB = q.sel3(y, qfma(J.jB4, gu, qfma(J.jB5, gV, t2)) * F.idB);
  gC = qfma(J.jC1, gB, qfma(J.jC2, gu, qfma(J.jC3, gV, rC))) * F.gh;
}

// One Kaps-Rentrop step attempt from s (its k1*, a1, e1 must hold ode_f at s, J the Jacobian there).
// Returns the mean square of the scaled error estimate; the new state comes back in yn*.
template <class Q>
SP_HD double quad_attempt_ros(const Q& q, const QuadCoef<Q>& c, const QuadState<Q>& s, const QuadJac<Q>& J, double hh,
                              double rtol, double atol, double fast_w, typename Q::T& ynA, typename Q::T& ynB,
                              typename Q::T& accn) {
  using namespace ros;
  using T = typename Q::T;
  QuadLU<Q> F;
  quad_factor(q, J, hh, F);
  const double ih = sp_rcp(hh);
  T g1A, g1B, g1C, g2A, g2B, g2C, g3A, g3B, g3C, g4A, g4B, g4C, fA, fB, fC, ee;
  quad_solve(q, J, F, s.k1A, s.k1B, s.a1, g1A, g1B, g1C);
  quad_rhs(q, c, qfma(A21, g1A, s.yA), qfma(A21, g1B, s.yB), fA, fB, fC, ee);
  quad_solve(q, J, F, qfma(C21 * ih, g1A, fA), qfma(C21 * ih, g1B, fB), qfma(C21 * ih, g1C, fC), g2A, g2B, g2C);
  quad_rhs(q, c, qfma(A32, g2A, qfma(A31, g1A, s.yA)), qfma(A32, g2B, qfma(A31, g1B, s.yB)), fA, fB, fC, ee);
  quad_solve(q, J, F, qfma(C32 * ih, g2A, qfma(C31 * ih, g1A, fA)), qfma(C32 * ih, g2B, qfma(C31 * ih, g1B, fB)),
             qfma(C32 * ih, g2C, qfma(C31 * ih, g1C, fC)), g3A, g3B, g3C);
  quad_solve(q, J, F, qfma(C43 * ih, g3A, qfma(C42 * ih, g2A, qfma(C41 * ih, g1A, fA))),
             qfma(C43 * ih, g3B, qfma(C42 * ih, g2B, qfma(C41 * ih, g1B, fB))),
             qfma(C43 * ih, g3C, qfma(C42 * ih, g2C, qfma(C41 * ih, g1C, fC))), g4A, g4B, g4C);
  ynA = qfma(B4, g4A, qfma(B3, g3A, qfma(B2, g2A, qfma(B1, g1A, s.yA))));
  ynB = qfma(B4, g4B, qfma(B3, g3B, qfma(B2, g2B, qfma(B1, g1B, s.yB))));
  accn = qfma(B4, g4C, qfma(B3, g3C, qfma(B2, g2C, qfma(B1, g1C, s.acc))));
  const T eA = qfma(E4, g4A, qfma(E2, g2A, E1 * g1A));       // E3 = 0
  const T eB = qfma(E4, g4B, qfma(E2, g2B, E1 * g1B));
  const T ec = qfma(E4, g4C, qfma(E2, g2C, E1 * g1C));
  const T sA = q.sel3(s.e1, qmax(qabs(s.yA), qabs(ynA)));    // u is weighted like Qr (Qr at the start of the step)
  // fast_w (<= 1) relaxes the terms of the reach and of what it carries (u, Vr, the in-stream masses, the daily sums)
  const T wA = q.sel3(s.e1 * fast_w, q.pick(SP_SOIL_ERR_WEIGHT * SP_ROS_W_SOIL, SP_SOIL_ERR_WEIGHT * SP_ROS_W_SOIL, SP_ROS_W_VG, 1.0));
  const T qA = (eA * wA) * qrcp_fast(qfma(rtol, sA, atol));
  const T qB = (eB * fast_w) * qrcp_fast(qfma(rtol, qmax(qabs(s.yB), qabs(ynB)), atol));
  const T qc = (ec * fast_w) * qrcp_fast(qfma(rtol, qmax(qabs(s.acc), qabs(accn)), atol));
  const double en2 = q.first(q.sum(qfma(qA, qA, qfma(qB, qB, qc * qc)))) * (1.0 / 12.0);
  return (en2 == en2) ? en2 : INFINITY;
}

// Day-boundary state of a quad kept outside the registers (device: shared memory, one per quad).
struct QuadMem {
  Hot h;
  Cold c;
  DayAux aux;
  Flags fl;
  int pad;
};
static_assert(sizeof(QuadMem) == 57 * sizeof(double), "QuadMem: odd double stride keeps 64-bit quad accesses conflict-free");

// State of one item between two launches that integrate consecutive parts of its record (the cost pilot integrates
// the first days in member order; the main launch continues from there in cost order instead of repeating them).
struct QuadCarry {
  QuadMem qm;
  double yA[4], yB[4];        // slots A and B of the four lanes at midnight
  double hstep, snow_depth;
  unsigned n_steps, n_rej, n_rhs;
  int status;
};

// IO policy concept of the quad program (all calls are made by every lane of the quad unless stated):
//   void wait(int day);                          // block until forcing and upstream inputs of `day` exist
//   void forcing(int day, double& P, double& E, double& doy, double& T_air);
//   void upstream(int day, double (&us)[4]);
//   void emit(const Q& q, int day, const double (&y)[NL], double Vr, const double (&acc)[NA], const double (&non)[13],
//             const Cold& c);                    // called by every lane (device: the lanes share the work)
//   void publish(int day);                       // leader only, after the emit of every lane
//
// The whole record of one (member, sub-catchment) item: replaces model.py:491-724 for it.
// STIFF compiles the Rosenbrock path in (networks); without it every day takes the explicit pair (ensembles of one
// sub-catchment, where the reach rate constant stays below ~150 per day and the extra code would only cost registers).
template <bool STIFF, class Q, class IO>
SP_HD void run_quad(const Q& q, const double* mp, const double* sp, double A_qr0, int nc_last,
                    const ThreadOptions& opt, int n_days, bool valid, QuadMem& qm, IO& io, ThreadCounters& cnt,
                    int day_begin, const QuadCarry* carry_in, QuadCarry* carry_out, bool resume, bool hand_over) {
  // resume / hand_over say whether carry_in / carry_out are used.  They are separate arguments because the branches they
  // guard hold quad shuffles and barriers: the caller passes conditions that are provably warp-uniform (a kernel
  // parameter, a warp vote), which a comparison of the per-thread pointers with null is not.
  using T = typename Q::T;
  QuadCoef<Q> qc;
  QuadState<Q> s;
  double Kf;
  {
    Hot h; Cold c; Flags fl; double y0[NL];
    setup_thread(mp, sp, A_qr0, nc_last, opt.strict_quirks, opt.run_mode_cal, h, c, fl, y0, Kf);
    quad_static_coef(q, h, qc);
    const double Qr0 = y0[iQr];
    s.yA = q.pick(y0[iVsA], y0[iVsS], y0[iVg], log(Qr0));
    s.yB = q.pick(y0[iMsus], y0[iTDPr], y0[iPPr], reach_volume(h, Qr0));    // Vr0, :457-459
    if (q.leader()) { qm.h = h; qm.c = c; qm.fl = fl; }
    q.sync();
  }
  unsigned n_steps = 0, n_rej = 0, n_rhs = 0;
#if defined(SP_LAT_PROBE) && defined(__CUDA_ARCH__)
  LatProbe lp = {};
  lp.t = clock64();
#endif
#ifdef SP_TIMELINE
  unsigned sp_lockstep_iters = 0;
#endif
  int status = 0;
  double snow_depth = mp[SIMPLYP_P_D_SNOW_0];       // only used with snow_on_device
  const double T1 = opt.step_len;
  double hstep = 0.05 * T1;
  if (resume) {                                     // continue a record: everything that crosses midnight
    s.yA = q.pick(carry_in->yA[0], carry_in->yA[1], carry_in->yA[2], carry_in->yA[3]);
    s.yB = q.pick(carry_in->yB[0], carry_in->yB[1], carry_in->yB[2], carry_in->yB[3]);
    hstep = carry_in->hstep;
    snow_depth = carry_in->snow_depth;
    n_steps = carry_in->n_steps; n_rej = carry_in->n_rej; n_rhs = carry_in->n_rhs; status = carry_in->status;
    if (q.leader()) qm = carry_in->qm;
    q.sync();
  }

  for (int day = day_begin; day < n_days; ++day) {
    // ---- start of the day: pre-ODE algebra (:497-618) -----------------------------------------
    io.wait(day);
    {
      Hot h = qm.h;
      double P, E, doy, T_air, us[4];
      io.forcing(day, P, E, doy, T_air);
      if (opt.snow_on_device) P = snow_day(P, T_air, mp[SIMPLYP_P_F_DDSM], snow_depth);
      io.upstream(day, us);
      DayAux aux;
      begin_day(mp, sp, qm.c, qm.fl, opt.dynamic_epc0, opt.dynamic_erod, P, E, doy, us, h, aux);
      quad_daily_coef(q, h, qc);
      q.sync();                                   // everybody has read qm before the leader rewrites it
      if (q.leader()) { qm.h = h; qm.aux = aux; }
      q.sync();                                   // ... and the end-of-day code of every lane sees the new values
    }
    s.acc = q.splat(0.0);                         // :618
    QuadJac<Q> J;
    quad_rhs_jac(q, qc, s.yA, s.yB, s.k1A, s.k1B, s.a1, s.e1, J);
    n_rhs += 1;
    // reach rate constant -d(du/dt)/du = Qr/((1-b_Q) Vr), per day: stiff days go to the Rosenbrock path
    const bool stiff = STIFF && (0.0 - q.first(q.bcast(J.dAA, 3))) > SP_STIFF_RATE;
    // Tolerance of the day (explicit pair): a local error of the reach and its in-stream masses is damped at the
    // reach's rate constant, so what reaches the daily flows and concentrations is the error committed per unit
    // time divided by that rate — measured on the bench ensemble, the worst daily error of a member falls as
    // 1/rate at a fixed tolerance.  The tolerance therefore grows in proportion to the rate above SP_TOL_RATE0 per
    // day (at most SP_TOL_GMAX-fold): the same worst error against the oracle, 11 % fewer attempts on average and
    // 20 % fewer for the members with the fastest reaches, which are the longest chains of a launch.
    // The record's first day is not relaxed: its in-stream masses start from zero (:441) and the day's fluxes are
    // the build-up itself, not a balance with the inputs that damps the local errors (a fast reach at a vertex of the
    // prior box reached 1.2e-5 on its first day at the relaxed tolerance, tests/test_box_vertices_cpu.py).
    double tol_inv2, day_rate;
    {
      const double rate = 0.0 - q.first(q.bcast(J.dAA, 3));
      day_rate = rate;
      double g = day == 0 ? 1.0 : sp_min(sp_max(rate * (1.0 / SP_TOL_RATE0), 1.0), SP_TOL_GMAX);
      if (stiff) g = sp_min(sp_max(rate * (1.0 / SP_ROS_RATE0), 1.0), SP_ROS_GMAX);
      tol_inv2 = stiff ? sp_rcp(g) : sp_rcp(g * g);        // stiff days: weight of the fast terms inside the norm
    }
    bool jac_fresh = true;
    double t = 0.0;
    int day_steps = 0;
    bool grow_ok = true;
    bool active = true;
    hstep = sp_min(hstep * SP_DAYSTART_FAC, T1);  // the forcing jumps at midnight
    if (stiff) hstep = sp_min(hstep, SP_H0_STIFF_C * sp_rcp(day_rate));
    // hstep * 1.0000001 (the test for the day's last step), carried beside hstep: after an accepted step it is formed
    // from the new step beside the comparison that chooses it, not after it, off the controller's dependent path (the
    // network builds, STIFF, form it from hstep where it is used: their 3-blocks build would spill the extra register)
    double hlim = hstep * 1.0000001;
    SP_LAT_MARK(LP_START);

    // ---- step loop: lock-step over the quads of a warp ------------------------------------------
    while (q.any(active)) {
#ifdef SP_LOOP_SYNCWARP
      q.sync();
#endif
#ifdef SP_TIMELINE
      ++sp_lockstep_iters;                        // analysis builds: attempts the WARP executed (lock-step)
#endif
      const double rem = T1 - t;
      const bool last = (STIFF ? hstep * 1.0000001 : hlim) >= rem;   // (networks: one register fewer, no spill)
      const double hh = active ? (last ? rem : hstep) : hstep;
      const bool do_rk = active && !stiff, do_ros = active && stiff;
      T ynA, ynB, accn;
      double en2 = 0.0, expo = -0.1;
      if (!STIFF || q.any(do_rk) || !q.any(do_ros)) {
        T k7A, k7B, a7, e7;
        const double e2 = quad_attempt(q, qc, s, hh, opt.rtol, opt.atol, ynA, ynB, accn, k7A, k7B, a7, e7 SP_LAT_ARG);
        SP_LAT_MARK(LP_ERR);
        if (do_rk) {
          en2 = e2 * tol_inv2;
          n_rhs += 6;
          if (en2 <= 1.0 || day_steps + 1 >= opt.max_steps_per_day || hh < 1e-12 * T1) {   // will be accepted below
            s.k1A = k7A; s.k1B = k7B; s.a1 = a7; s.e1 = e7;
          }
        }
      }
      if (STIFF && q.any(do_ros)) {
        if (q.any(do_ros && !jac_fresh)) {         // ode_f and its Jacobian at the state reached by the last step
          T fA, fB, fC, e0;
          QuadJac<Q> Jn;
          quad_rhs_jac(q, qc, s.yA, s.yB, fA, fB, fC, e0, Jn);
          if (do_ros && !jac_fresh) {
            s.k1A = fA; s.k1B = fB; s.a1 = fC; s.e1 = e0;
            J = Jn;
            jac_fresh = true;
            n_rhs += 1;
          }
        }
        T rA, rB, rC;
        const double e2 = quad_attempt_ros(q, qc, s, J, hh, opt.rtol * SP_ROS_TOL_SCALE, opt.atol * SP_ROS_TOL_SCALE,
                                           last ? 1.0 : tol_inv2, rA, rB, rC);
        if (do_ros) { en2 = e2; expo = -0.125; ynA = rA; ynB = rB; accn = rC; n_rhs += 2; }
      }
      if (active) {
        n_steps += 1;
        day_steps += 1;
        bool accept = en2 <= 1.0;
        if (!accept && (day_steps >= opt.max_steps_per_day || hh < 1e-12 * T1)) {
          accept = true;                          // forward-progress guard
          status |= 1;
        }
        // the factor's cap (1 after a rejection and on the step after one) is known before the factor: it is applied
        // inside the fp32 clamp instead of as a double min after it
        const double fac = step_factor_sq(en2, expo, (accept && grow_ok) ? SP_CTRL_MAXGROW : 1.0);
#ifdef SP_ATTEMPT_HOOK
        SP_ATTEMPT_HOOK(io, day, day_steps, t, hh, en2, accept);   // analysis builds only (scripts/)
#endif
        if (accept) {
          t += hh;
          s.yA = ynA; s.yB = ynB; s.acc = accn;
          if (stiff) jac_fresh = false;           // (the explicit path took its FSAL derivative above)
          grow_ok = true;
          const double hnew = hh * fac;
          const bool keep = last && hnew < hstep;
          hlim = keep ? hlim : hnew * 1.0000001;
          hstep = keep ? hstep : hnew;
          if (last) active = false;
        } else {
          n_rej += 1;
          hstep = hh * fac;
          hlim = hstep * 1.0000001;
          grow_ok = false;
        }
      }
      SP_LAT_MARK(LP_CTRL);
      SP_LAT_COUNT(LP_ITERS);
    }

    // ---- end of the day: post-ODE algebra (:643-724), output --------------------------------------
#ifdef SP_DAY_HOOK
    SP_DAY_HOOK(io, day, n_steps);                // analysis builds only (scripts/): per-day attempt counts
#endif
    {
      double y[NL], yraw[NL], acc[NA], non[13];
      const double u_end = q.first(q.bcast(s.yA, 3));
      y[iVsA] = q.first(q.bcast(s.yA, 0)); y[iVsS] = q.first(q.bcast(s.yA, 1)); y[iVg] = q.first(q.bcast(s.yA, 2));
      y[iQr] = sp_exp(u_end);
      y[iMsus] = q.first(q.bcast(s.yB, 0)); y[iTDPr] = q.first(q.bcast(s.yB, 1)); y[iPPr] = q.first(q.bcast(s.yB, 2));
      const double Vr = q.first(q.bcast(s.yB, 3));
      acc[1] = q.first(q.bcast(s.acc, 0)); acc[2] = q.first(q.bcast(s.acc, 1)); acc[3] = q.first(q.bcast(s.acc, 2));
      acc[0] = q.first(q.bcast(s.acc, 3));
      bool finite = (Vr - Vr == 0.0);
#pragma unroll
      for (int i = 0; i < NL; ++i) { yraw[i] = y[i]; finite = finite && (y[i] - y[i] == 0.0); }
      if (!finite) status |= 2;
      Cold c = qm.c;
      const Hot& h = qm.h;
      end_day(h, c, qm.fl, opt.dynamic_epc0, qm.aux, y, non);
      s.yA = q.pick(y[iVsA], y[iVsS], y[iVg], u_end);          // groundwater floor moved Vg (:670)
      // Vr - L/(a_Q 86400) Qr^(1-b_Q) is conserved by ode_f (:127-131) and zero initially (:457-459): an error
      // along that direction is never damped and would random-walk over a 30-year record, so the volume carried
      // into the next day is put back on the curve (the reported Vr is the integrated one).
      s.yB = q.pick(y[iMsus], y[iTDPr], y[iPPr], sp_exp((1.0 - h.bQ) * u_end) * sp_rcp(h.cR));
      if (valid) io.emit(q, day, yraw, Vr, acc, non, c);   // by every lane: the lanes share the row / the series
      q.sync();                                   // every lane has read qm.c (above) and stored its part of the row
      if (q.leader()) {                           // before the leader rewrites qm.c and publishes the day
        qm.c = c;
        if (valid) io.publish(day);
      }
      q.sync();                                   // tomorrow's begin_day of every lane reads the new qm.c
    }
    SP_LAT_MARK(LP_END);
    SP_LAT_COUNT(LP_DAYS);
  }
  if (hand_over) {
    const double a0 = q.first(q.bcast(s.yA, 0)), a1 = q.first(q.bcast(s.yA, 1)), a2 = q.first(q.bcast(s.yA, 2)),
                 a3 = q.first(q.bcast(s.yA, 3));
    const double b0 = q.first(q.bcast(s.yB, 0)), b1 = q.first(q.bcast(s.yB, 1)), b2 = q.first(q.bcast(s.yB, 2)),
                 b3 = q.first(q.bcast(s.yB, 3));
    if (q.leader() && valid) {
      carry_out->qm = qm;
      carry_out->yA[0] = a0; carry_out->yA[1] = a1; carry_out->yA[2] = a2; carry_out->yA[3] = a3;
      carry_out->yB[0] = b0; carry_out->yB[1] = b1; carry_out->yB[2] = b2; carry_out->yB[3] = b3;
      carry_out->hstep = hstep;
      carry_out->snow_depth = snow_depth;
      carry_out->n_steps = n_steps; carry_out->n_rej = n_rej; carry_out->n_rhs = n_rhs; carry_out->status = status;
    }
  }
  cnt.steps = n_steps;
  cnt.rejected = n_rej;
#ifdef SP_TIMELINE
  cnt.rejected = sp_lockstep_iters;
#endif
  cnt.rhs_evals = n_rhs;
  cnt.status = status;
#if defined(SP_LAT_PROBE) && defined(__CUDA_ARCH__)
  for (int i = 0; i < LP_N; ++i) cnt.lat[i] = lp.acc[i];
#endif
  (void)Kf;
}


// The whole record, or a part of it continued from / handed over to a stored midnight state (host builds, tests).
template <bool STIFF, class Q, class IO>
SP_HD void run_quad(const Q& q, const double* mp, const double* sp, double A_qr0, int nc_last,
                    const ThreadOptions& opt, int n_days, bool valid, QuadMem& qm, IO& io, ThreadCounters& cnt,
                    int day_begin = 0, const QuadCarry* carry_in = nullptr, QuadCarry* carry_out = nullptr) {
  run_quad<STIFF>(q, mp, sp, A_qr0, nc_last, opt, n_days, valid, qm, io, cnt, day_begin, carry_in, carry_out,
                  carry_in != nullptr, carry_out != nullptr);
}

}  // namespace simplyp
