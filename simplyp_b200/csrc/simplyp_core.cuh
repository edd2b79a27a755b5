// simplyp_core.cuh — per-(member, sub-catchment) arithmetic of the SimplyP v0-2A daily step.
//
// Everything here is inline __host__ __device__ code operating on named scalars / fixed-size
// arrays with compile-time indices, so that under nvcc the whole Runge–Kutta state lives in
// registers.  The same header is compiled for the host ONLY by tests/hostemu (a test harness
// that lets the CPU-only test tier exercise this arithmetic); the product library
// (simplyp_kernels.cu) has no host execution path.
//
// Reference map (all line numbers: Current_Release/v0-2A/simplyP/model.py):
//   gate()            f_x                         :23-37
//   soilp_update()    discretized_soilP           :39-56
//   (ode_f itself, :58-187, is quad_rhs() in simplyp_quad.cuh)
//   setup_thread()    run_simply_p, setup part    :318-335, :349, :377-463, :469
//   begin_day()       run_simply_p, pre-ODE part  :497-501, :549-594, :600-611, :618
//   kRK, step_factor_sq()  tableau and controller of the embedded pair that replaces scipy.integrate.odeint, :640
//   end_day()         run_simply_p, post-ODE part :643-724
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../include/simplyp_b200.h"

#if defined(__CUDACC__)
#define SP_HD __host__ __device__ __forceinline__
#else
#define SP_HD inline
#endif

namespace simplyp {

// ------------------------------------------------------------------------------------------
// number of live ODE states and of daily accumulators (ode_f's y[0..11] split by role)
//   live: VsA VsS Vg Vr Qr Msus TDPr PPr      (y[0..4], y[6], y[8], y[10])
//   acc : Qr_av Msus_out TDPr_out PPr_out     (y[5], y[7], y[9], y[11]); zero at day start (:618)
//   The day-boundary code exchanges Qr (not the quad program's u = ln Qr); the reach volume follows
//   Vr == L/(a_Q*86400)*Qr^(1-b_Q), which ode_f's dVr/dt = net and dQr/dt = net*a_Q*Qr^b_Q*86400/((1-b_Q)*L)
//   (:127-131) conserve and the reference's initial condition (:457-459) satisfies (reach_volume()).
constexpr int NL = 7;
constexpr int NA = 4;
enum { iVsA = 0, iVsS, iVg, iQr, iMsus, iTDPr, iPPr };

// Constants of the RHS that are fixed within one day.  Kept in registers.
struct Hot {
  double fc, inv_fcd, mu, inv_TsA, inv_TsS, inv_Tg, Qg_min, inv_Qgd;
  double Pin, aE;        // P*(1-f_quick), alpha*PET
  double fA, fS, beta;
  double qin0;           // Qq + Qr_US
  double kQ, bQ, kM;     // a_Q*86400/((1-b_Q)*L_reach), b_Q, k_M
  double cR;             // a_Q*86400/L_reach: Qr/Vr = cR*Qr^b_Q
  double cM, MsusUS;     // sediment source coefficient, upstream sediment
  double tA, tS, tG, t0; // TDP: coefficients of QsA, QsS, Qg and the constant source
  double cP, PPUS;       // PP source coefficient, upstream PP
};

// Per-thread constants and the soil-P carry that are only touched at day boundaries.
// The CUDA kernels keep one of these per thread in shared memory (25 doubles: an odd stride,
// so that 64-bit accesses of a half-warp fall in distinct banks).
struct Cold {
  double f_quick, alpha;
  double A_catch;
  double KfMsoil;        // Kf*Msoil
  double inv_Msoil_EPP;  // E_PP/Msoil
  double P_inactive;
  double pnetA, pnetNC;  // P_netInput*A_catch*100/365 for A and NC land
  // sediment delivery: Esus_A = baseA*C_cover_A(day) with baseA = E_M*S_reach*S_Ar*(1-C_measures_A);
  // Esus_S, Esus_IG are constant (:591-594).  Folded with the land-use fractions they multiply:
  double m1, m2;         // cM = m1*C_A + m2            (f_Ar*baseA ; f_IG*Esus_IG + f_S*Esus_S)
  double pp1, pp2, pp3;  // old arable*C_A, old IG, old semi-natural (x P_inactive)   (:171-173)
  double pp4, pp5;       // newly-converted arable*C_A, newly-converted IG + SN        (:174-176)
  double tdpA, tdpNC;    // f_A(1-f_NC_A), f_A f_NC_A + f_S f_NC_S
  double tdp_fixed;      // TDPeff (kg/day)
  // soil-P state carried between days (:426-446, :684-715)
  double PlabA, TDPsA, PlabNC, TDPsNC, concA, concNC;
  double T_g;            // groundwater time constant (the floor resets Vg = Qg*T_g, :670)
};
static_assert(sizeof(Cold) == 25 * sizeof(double), "Cold must stay 25 doubles (bank-conflict-free stride)");

struct Flags {
  int nc_is_A;       // NC land takes arable hydrology inside ode_f (:113)
  int nc_is_S;       // NC land is semi-natural (:429, :608)
  int post_nc_is_A;  // which hydrology the post-ODE soil-P step uses (:442, :676; leaked variable)
};

// Run options and per-item counters shared by the kernels and the program (SimplypOptions, narrowed).
struct ThreadOptions {
  double rtol, atol, step_len;
  int max_steps_per_day;
  int dynamic_epc0, dynamic_erod, run_mode_cal, strict_quirks;
  int snow_on_device;   // forcing carries raw precipitation and T_air, snow is a per-member scan
};

struct ThreadCounters {
  long long steps, rejected, rhs_evals;
  int status;
#ifdef SP_LAT_PROBE
  long long lat[8];     // analysis builds: SM cycles of the warp by section of the day loop (simplyp_quad.cuh, LatProbe)
#endif
};

// ------------------------------------------------------------------------------------------
SP_HD double sp_max(double a, double b) { return a > b ? a : b; }
SP_HD double sp_min(double a, double b) { return a < b ? a : b; }

// ---- branch-free fp64 elementary functions for the ranges this model visits -------------------
// The CUDA math library's exp/log/division carry special-case branches (and, for division, a
// call to a slow path) that cost issue slots and registers in a kernel whose critical path is one
// long dependent fp64 chain.  These versions assume finite, normal arguments (|x| < 700 for exp,
// x > 0 for log, normal divisor) — a NaN still propagates as NaN, which the step control rejects.
// Polynomials are evaluated with Estrin's scheme (short dependency chains).  Accuracy ~1-2 ulp.
SP_HD long long sp_d2ll(double x) {
#if defined(__CUDA_ARCH__)
  return __double_as_longlong(x);
#else
  long long b; memcpy(&b, &x, 8); return b;
#endif
}
SP_HD double sp_ll2d(long long b) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double(b);
#else
  double x; memcpy(&x, &b, 8); return x;
#endif
}

SP_HD double sp_rcp(double x) {
#if defined(__CUDA_ARCH__)
  double r;
  // volatile: keeps the MUFU where the source puts it relative to the quad broadcasts (ptxas otherwise sinks the
  // whole reciprocal chain behind the exponential and puts it on the critical path of the RHS evaluation)
  asm volatile("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));   // ~20 good bits
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  return r;
#else
  return 1.0 / x;
#endif
}

// a / b given rb = 1/b to (nearly) full precision: product, exact remainder by fma, one correction.  Branch-free and
// call-free; equal to the IEEE quotient except in rare last-bit cases.
SP_HD double sp_div(double a, double b, double rb) {
#if defined(__CUDA_ARCH__)
  const double q = a * rb;
  return fma(fma(-b, q, a), rb, q);
#else
  (void)rb;
  return a / b;
#endif
}

// 1/x to ~40 bits (one Newton step on the 20-bit hardware seed): for the reciprocal INSIDE the RHS evaluation, whose
// accuracy requirement is the integration tolerance (1e-7), not the last bit.
SP_HD double sp_rcp40(double x) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  return fma(r, fma(-x, r, 1.0), r);
#else
  return 1.0 / x;
#endif
}

// Polynomial coefficients live in constant memory on the device: a DFMA can take a constant-bank operand
// directly, whereas a 64-bit literal costs two extra move instructions every time it is rematerialised
// (and with ~250 live registers the compiler rematerialises all of them inside the step loop).
#if defined(__CUDA_ARCH__)
#define SP_CONST __constant__
#else
#define SP_CONST static const
#endif
SP_CONST double kExpC[16] = {
    1.4426950408889634074, -6.93147180369123816490e-01, -1.90821492927058770002e-10,
    1.0 / 6.0, 0.5, 1.0 / 120.0, 1.0 / 24.0, 1.0 / 5040.0, 1.0 / 720.0, 1.0 / 362880.0, 1.0 / 40320.0,
    1.0 / 39916800.0, 1.0 / 3628800.0, 1.0 / 479001600.0, 0.0, 0.0};
SP_CONST double kLogC[16] = {
    1.0 / 3.0, 1.0 / 7.0, 1.0 / 5.0, 1.0 / 11.0, 1.0 / 9.0, 1.0 / 15.0, 1.0 / 13.0, 1.0 / 19.0, 1.0 / 17.0,
    1.0 / 21.0, 6.93147180369123816490e-01, 1.90821492927058770002e-10, 1.4142135623730951, 0.0, 0.0, 0.0};

// ~7 significant digits: only for the error norm and the step-size factor
SP_HD double sp_rcp_fast(double x) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  return fma(r, fma(-x, r, 1.0), r);
#else
  return 1.0 / x;
#endif
}

// e^x for |x| < 700, no range check (the RHS arguments -mu*Vs, b_Q*ln Qr, k_M*ln Qr are far inside).
SP_HD double sp_exp_core(double x) {
  // x = k ln2 + r, |r| <= ln2/2 ; e^r by its degree-12 Taylor polynomial (remainder < 2e-16)
  const double kf = rint(x * kExpC[0]);
  double r = fma(kf, kExpC[1], x);
  r = fma(kf, kExpC[2], r);
  const double r2 = r * r, r4 = r2 * r2, r8 = r4 * r4;
  const double p01 = 1.0 + r;
  const double p23 = fma(r, kExpC[3], kExpC[4]);
  const double p45 = fma(r, kExpC[5], kExpC[6]);
  const double p67 = fma(r, kExpC[7], kExpC[8]);
  const double p89 = fma(r, kExpC[9], kExpC[10]);
  const double pab = fma(r, kExpC[11], kExpC[12]);
  const double q0 = fma(r2, p23, p01);          // terms 0..3
  const double q1 = fma(r2, p67, p45);          // terms 4..7  (times r^4)
  const double q2 = fma(r2, pab, p89);          // terms 8..11 (times r^8)
  const double lo = fma(r4, q1, q0);
  const double hi = fma(r4, kExpC[13], q2);     // 1/12! carries r^12 = r^8 * r^4
  const double p = fma(r8, hi, lo);
  // scale by 2^k through the exponent field
  return sp_ll2d(sp_d2ll(p) + ((long long)kf << 52));
}

// Table-driven e^x for the quad kernel: x = (64 m + j) ln2/64 + r with |r| <= ln2/128, e^x = 2^m * 2^(j/64) * e^r.
// The reduction uses the 1.5*2^52 trick (the integer lands in the low word of the sum: no FRND/F2I), e^r is a
// degree-4 polynomial (remainder r^5/5! < 4e-14: far below the integration tolerance this function serves) and 2^(j/64) comes from a 64-entry table (`tab`: shared memory on
// the device, kExp2Tab on the host).  The table entry is scaled by 2^m with integer arithmetic while the
// polynomial is still being evaluated, so one multiply finishes the function.  |x| < 700, no range check.
// Relative accuracy 4e-14.
constexpr int EXP_TAB = 64;
SP_CONST double kExpT[12] = {
    92.33248261689366,      // 64/ln2
    -0.010830424696249145,   // -ln2/64 (nearest double)
    0.0,                     // (unused)
    6755399441055744.0,      // 1.5*2^52
    0.5, 1.0 / 6.0, 1.0 / 24.0, 1.0 / 120.0, 0.0, 0.0, 0.0, 0.0};
// 2^(j/64), j = 0..63, correctly rounded (generated with 60-digit decimal arithmetic)
SP_CONST double kExp2Tab[EXP_TAB] = {
    1.0, 1.0108892860517005, 1.0218971486541166, 1.0330248790212284,
    1.0442737824274138, 1.0556451783605572, 1.0671404006768237, 1.0787607977571199,
    1.0905077326652577, 1.102382583307841, 1.1143867425958924, 1.1265216186082418,
    1.1387886347566916, 1.1511892299529827, 1.1637248587775775, 1.1763969916502812,
    1.189207115002721, 1.202156731452703, 1.215247359980469, 1.22848053610687,
    1.241857812073484, 1.255380757024691, 1.2690509571917332, 1.2828700160787783,
    1.2968395546510096, 1.3109612115247644, 1.3252366431597413, 1.339667524053303,
    1.3542555469368927, 1.3690024229745905, 1.383909881963832, 1.3989796725383112,
    1.4142135623730951, 1.42961333839197, 1.4451808069770467, 1.460917794180647,
    1.4768261459394993, 1.4929077282912648, 1.5091644275934228, 1.5255981507445384,
    1.5422108254079407, 1.559004400237837, 1.5759808451078865, 1.593142151342267,
    1.6104903319492543, 1.6280274218573478, 1.645755478153965, 1.6636765803267364,
    1.681792830507429, 1.7001063537185235, 1.718619298122478, 1.7373338352737062,
    1.7562521603732995, 1.7753764925265212, 1.7947090750031072, 1.8142521755003989,
    1.8340080864093424, 1.8539791250833855, 1.8741676341103, 1.8945759815869656,
    1.9152065613971474, 1.9360617934922943, 1.9571441241754002, 1.978456026387951};
// `t` = x*(64/ln2) + 1.5*2^52 may be formed by the caller.
SP_HD double sp_exp_tab_pre(double x, double t, const double* tab) {
  const double kf = t - kExpT[3];
  const int ki = (int)(unsigned)(sp_d2ll(t) & 0xffffffffLL);      // two's-complement integer in the low word
  // 2^(j/64) * 2^m: exponent field of the table entry plus m (off the critical path)
#if defined(__CUDA_ARCH__)
  // on the high word only: (m << 20) = (ki with its low 6 bits cleared) << 14 — three integer instructions instead of
  // a 64-bit add with carry
  const double tj = tab[ki & (EXP_TAB - 1)];
  const double sc = __hiloint2double(__double2hiint(tj) + (int)(((unsigned)ki & ~(unsigned)(EXP_TAB - 1)) << 14),
                                     __double2loint(tj));
#else
  const double sc = sp_ll2d(sp_d2ll(tab[ki & (EXP_TAB - 1)]) + ((long long)(ki >> 6) << 52));
#endif
  // one FMA reduces the argument: the product is exact inside the FMA, so the only error is |k| times the rounding
  // of the constant ln2/64 (1.2e-18): 3e-15 for the largest arguments of the RHS (k_M ln Qr ~ 26), 8e-14 at |x| = 700
  const double r = fma(kf, kExpT[1], x);
  const double r2 = r * r;
  const double b = fma(r, kExpT[5], kExpT[4]);
  const double p = fma(r2, fma(r2, kExpT[6], b), r);              // e^r - 1 = r + r^2/2 + r^3/6 + r^4/24
  return fma(sc, p, sc);
}
SP_HD double sp_exp_tab(double x, const double* tab) { return sp_exp_tab_pre(x, fma(x, kExpT[0], kExpT[3]), tab); }

// Range-checked variant for the once-a-day algebra: arguments are clamped to [-700, 700]
// (e^-700 ~ 1e-304 stands in for an underflow to 0).
SP_HD double sp_exp(double x) { return sp_exp_core(sp_min(sp_max(x, -700.0), 700.0)); }

SP_HD double sp_log(double x) {
  // x = 2^e * m, m in [sqrt(1/2), sqrt(2)); log m = 2 atanh(f), f = (m-1)/(m+1), |f| <= 0.1716
  long long b = sp_d2ll(x);
  long long e = ((b >> 52) & 0x7ff) - 1023;
  b = (b & 0x000fffffffffffffLL) | 0x3ff0000000000000LL;
  double m = sp_ll2d(b);
  if (m > kLogC[12]) { m *= 0.5; e += 1; }
  const double f = (m - 1.0) * sp_rcp(m + 1.0);
  const double s = f * f, s2 = s * s, s4 = s2 * s2, s8 = s4 * s4;
  // 1 + s/3 + s^2/5 + ... + s^10/21
  const double a01 = fma(s, kLogC[0], 1.0);
  const double a23 = fma(s, kLogC[1], kLogC[2]);
  const double a45 = fma(s, kLogC[3], kLogC[4]);
  const double a67 = fma(s, kLogC[5], kLogC[6]);
  const double a89 = fma(s, kLogC[7], kLogC[8]);
  const double c0 = fma(s2, a23, a01);
  const double c1 = fma(s2, a67, a45);
  const double c2 = fma(s2, kLogC[9], a89);
  const double poly = fma(s8, c2, fma(s4, c1, c0));
  const double ed = (double)e;
  return fma(ed, kLogC[10], fma(2.0 * f, poly, ed * kLogC[11]));
}

// f_x(x, thr, 0.01) expressed on u = (x-thr)/(thr*0.01): 0 for u<0, 1 for u>1, 3u^2-2u^3 between.
SP_HD double sp_clamp01(double u) {
#if defined(__CUDA_ARCH__)
  // decided on the high word with integer compares: no fp64-pipe DSETP and none of the NaN fix-ups the
  // compiler attaches to the min/max idiom (u is finite here; a NaN passes through and the step is rejected)
  const int hi = __double2hiint(u);
  const double z = (hi < 0) ? 0.0 : u;
  return (hi >= 0x3ff00000) ? 1.0 : z;
#else
  return sp_min(sp_max(u, 0.0), 1.0);
#endif
}
SP_HD double gate(double u) {
  u = sp_clamp01(u);
  return u * u * fma(-2.0, u, 3.0);
}

// Reach volume on the invariant curve (reported as the 'Vr' output column).
SP_HD double reach_volume(const Hot& c, double Qr) { return Qr / (c.cR * sp_exp(c.bQ * sp_log(Qr))); }

// ------------------------------------------------------------------------------------------
// discretized_soilP (:39-56).  pnet = P_netInput*A_catch*100/365.
SP_HD void soilp_update(double pnet, double KfMsoil, double EPC0, double Qs, double Qq, double Vs,
                        double& TDPs, double& Plab) {
  const double a = pnet + KfMsoil * EPC0;
  const double iVs = sp_rcp(Vs);
  const double b = (KfMsoil + Qs + Qq) * iVs;
  const double ib = sp_rcp(b);
  const double ab = a * ib;
  const double e = sp_exp(-b);
  TDPs = ab + (TDPs - ab) * e;                                   // :44
  double sorp = 0.0;
  if (Vs > 0.0) {                                                // :50
    const double ab0 = ab * iVs;                                 // a/(b*Vs)
    sorp = KfMsoil * (ab0 - EPC0 + ib * (TDPs * iVs - ab0) * (1.0 - e));   // :51 (updated TDPs)
  }
  Plab = Plab + sorp;                                            // :54
}

// Dynamic arable crop-cover factor (:354-361, :563-580), triangular wave around the two
// erosion-risk mid-points; `dayNo in np.arange(start, end)` is reproduced literally.
SP_HD double season_cover(double doy, double mid, double C_cover) {
  const double half = 30.0;  // E_risk_period/2
  const double start = mid - half, end = mid + half;
  const double k = doy - start;
  const bool inside = (k >= 0.0) && (doy < end) && (k == floor(k));
  if (inside) {
    // lin_interp (helper_functions.py:77) over windows that are exactly half = 30 days wide
    if (doy < mid) return C_cover + (1.0 - C_cover) * (doy - start) * (1.0 / half);
    return 1.0 + (C_cover - 1.0) * (doy - mid) * (1.0 / half);
  }
  return C_cover - (1.0 - C_cover) * (60.0 / (2.0 * (365.0 - 60.0)));
}

// ------------------------------------------------------------------------------------------
// One-off setup of a (member, sub-catchment) thread: derived parameters and initial conditions.
//   mp      : member parameter row [SIMPLYP_NP_MEMBER]
//   sp      : this sub-catchment's parameter row [SIMPLYP_NP_SC]
//   A_qr0   : A_catch of the sub-catchment p['SC_Qr0'] (:386)
//   nc_last : NC type of the LAST sub-catchment in run order (0 none, 1 'A', 2 'S'), for the
//             leaked-variable quirk; pass this SC's own type to disable it
SP_HD void setup_thread(const double* mp, const double* sp, double A_qr0, int nc_last, int strict_quirks,
                        int run_mode_cal, Hot& h, Cold& c, Flags& fl, double (&y)[NL], double& Kf_out) {
  const double A = sp[SIMPLYP_SC_A_CATCH];
  const double fAr = sp[SIMPLYP_SC_F_AR], fIG = sp[SIMPLYP_SC_F_IG], fS = sp[SIMPLYP_SC_F_S];
  const double fNCAr = sp[SIMPLYP_SC_F_NC_AR], fNCIG = sp[SIMPLYP_SC_F_NC_IG], fNCS = sp[SIMPLYP_SC_F_NC_S];
  const double fA = fIG + fAr;                                   // :318
  const double fNCA = fAr * fNCAr + fNCIG * fIG;                 // :319
  int nc = 0;                                                    // :325-334
  if (fNCA > 0.0) nc = 1; else if (fNCS > 0.0) nc = 2;
  fl.nc_is_A = (nc == 1);
  fl.nc_is_S = (nc == 2);
  fl.post_nc_is_A = strict_quirks ? (nc_last == 1) : (nc == 1);

  const double fc = mp[SIMPLYP_P_FC];
  h.fc = fc;
  h.inv_fcd = 1.0 / (fc * 0.01);
  h.mu = -log(0.01) / fc;                                        // :349
  h.inv_TsA = 1.0 / mp[SIMPLYP_P_TS_A];
  h.inv_TsS = 1.0 / mp[SIMPLYP_P_TS_S];
  h.inv_Tg = 1.0 / mp[SIMPLYP_P_T_G];
  h.Qg_min = mp[SIMPLYP_P_QG_MIN];
  h.inv_Qgd = 1.0 / (h.Qg_min * 0.01);
  h.fA = fA;
  h.fS = fS;
  h.beta = mp[SIMPLYP_P_BETA];
  const double aQ = mp[SIMPLYP_P_A_Q], bQ = mp[SIMPLYP_P_B_Q];
  h.kQ = aQ * 86400.0 / ((1.0 - bQ) * sp[SIMPLYP_SC_L_REACH]);   // :130
  h.cR = aQ * 86400.0 / sp[SIMPLYP_SC_L_REACH];
  h.bQ = bQ;
  h.kM = mp[SIMPLYP_P_K_M];
  h.tG = mp[SIMPLYP_P_TDPG] * A;                                 // UC_Cinv(TDPg, A_catch), :163
  h.Pin = h.aE = h.qin0 = h.cM = h.MsusUS = h.tA = h.tS = h.t0 = h.cP = h.PPUS = 0.0;

  c.f_quick = mp[SIMPLYP_P_F_QUICK];
  c.alpha = mp[SIMPLYP_P_ALPHA];
  c.A_catch = A;
  const double Msoil = mp[SIMPLYP_P_MSOIL_M2] * 1e6 * A;         // :404
  c.P_inactive = 1e-6 * mp[SIMPLYP_P_SOILP_S] * Msoil;           // :407
  const double EPC0_0_A = mp[SIMPLYP_P_EPC0_A] * A;              // :412
  const double EPC0_0_S = mp[SIMPLYP_P_EPC0_S] * A;
  const double Plab0_A = 1e-6 * (mp[SIMPLYP_P_SOILP_A] - mp[SIMPLYP_P_SOILP_S]) * Msoil;   // :415
  const double TDPs0_A = EPC0_0_A * fc;                          // :420 (VsA0 = fc)
  double Kf;
  if (run_mode_cal) Kf = 1e-6 * (mp[SIMPLYP_P_SOILP_A] - mp[SIMPLYP_P_SOILP_S]) / EPC0_0_A;   // :451
  else Kf = mp[SIMPLYP_P_KF];
  Kf_out = Kf;
  c.KfMsoil = Kf * Msoil;
  c.inv_Msoil_EPP = mp[SIMPLYP_P_E_PP] / Msoil;
  c.pnetA = mp[SIMPLYP_P_PNET_A] * A * 100.0 / 365.0;            // :42
  c.pnetNC = mp[SIMPLYP_P_PNET_NC] * A * 100.0 / 365.0;
  const double EM_Sr = mp[SIMPLYP_P_E_M] * sp[SIMPLYP_SC_S_REACH];           // :591-594
  const double baseA = EM_Sr * sp[SIMPLYP_SC_S_AR] * (1.0 - mp[SIMPLYP_P_CMEAS_A]);
  const double eS = EM_Sr * sp[SIMPLYP_SC_S_SN] * mp[SIMPLYP_P_CCOVER_S] * (1.0 - mp[SIMPLYP_P_CMEAS_S]);
  const double eIG = EM_Sr * sp[SIMPLYP_SC_S_IG] * mp[SIMPLYP_P_CCOVER_IG] * (1.0 - mp[SIMPLYP_P_CMEAS_IG]);
  c.m1 = fAr * baseA;                                            // :141
  c.m2 = fIG * eIG + fS * eS;                                    // :142-143
  c.pp1 = fAr * (1.0 - fNCAr) * baseA;                           // :171
  c.pp2 = fIG * (1.0 - fNCIG) * eIG;                             // :172
  c.pp3 = fS * (1.0 - fNCS) * eS * c.P_inactive;                 // :173
  c.pp4 = fAr * fNCAr * baseA;                                   // :174
  c.pp5 = fIG * fNCIG * eIG + fS * fNCS * eS;                    // :175-176
  c.T_g = mp[SIMPLYP_P_T_G];
  c.tdpA = fA * (1.0 - fNCA);                                    // :155,159
  c.tdpNC = fA * fNCA + fS * fNCS;                               // :156-157,160-161
  double TDPeff = sp[SIMPLYP_SC_TDPEFF];
  if (TDPeff != TDPeff) TDPeff = 0.0;                            // blank cell -> 0, :462-463
  c.tdp_fixed = TDPeff;

  // soil-P carry (:426-446)
  c.PlabA = Plab0_A;
  c.TDPsA = TDPs0_A;
  if (nc == 2) { c.PlabNC = Plab0_A; c.TDPsNC = TDPs0_A; }       // :429-431
  else { c.PlabNC = 0.0; c.TDPsNC = 0.0; }                       // :433-434 (TDPs0['S'] = 0)
  c.concA = TDPs0_A / fc;                                        // :438
  c.concNC = c.TDPsNC / fc;                                      // :446 (VsA0 == VsS0 == fc)
  (void)EPC0_0_S;

  // hydrology initial conditions (:377-390, :457-459)
  const double Qr0 = mp[SIMPLYP_P_QR0_INIT] * 86400.0 / (1000.0 * A_qr0);    // UC_Qinv, :386
  y[iVsA] = fc;
  y[iVsS] = fc;
  y[iVg] = mp[SIMPLYP_P_BETA] * Qr0 * mp[SIMPLYP_P_T_G];
  y[iQr] = Qr0;                                                  // Vr0 (:457-459) lies on the invariant curve
  y[iMsus] = 0.0;
  y[iTDPr] = 0.0;
  y[iPPr] = 0.0;
}

// snow_hydrol_inputs (inputs.py:159-210) for one day: precipitation falls as snow when T_air < 0, potential melt
// f_DDSM*T_air (>= 0) is limited by the pack at the start of the day; returns P = rain + melt and advances the pack.
SP_HD double snow_day(double precip, double t_air, double f_DDSM, double& depth) {
  const double p_snow = (t_air < 0.0) ? precip : 0.0;            // :183-185
  const double p_rain = precip - p_snow;                         // :186
  double melt_pot = f_DDSM * (t_air - 0.0);                      // :188
  if (melt_pot < 0.0) melt_pot = 0.0;                            // :191
  const double melt = sp_min(melt_pot, depth);                   // :203
  depth = depth + p_snow - melt;                                 // :204
  return p_rain + melt;                                          // :208
}

// Values of a day that end up in the output row but are not states.
struct DayAux {
  double Qq, C_cover_A, EPC0_A, EPC0_NC;
};

// Pre-ODE part of one day (:497-501, :549-611): fills the day-dependent members of Hot.
//   P, E, doy : forcing of the day;  us[4] : upstream Qr (already area-scaled), Msus, TDP, PP
SP_HD void begin_day(const double* mp, const double* sp, const Cold& c, const Flags& fl,
                     int dynamic_epc0, int dynamic_erod, double P, double E, double doy,
                     const double (&us)[4], Hot& h, DayAux& aux) {
  const double Qq = c.f_quick * P;                               // :501
  aux.Qq = Qq;
  h.Pin = P * (1.0 - c.f_quick);
  h.aE = c.alpha * E;
  h.qin0 = Qq + us[0];
  h.MsusUS = us[1];
  h.PPUS = us[3];
  // erodibility (:549-594)
  double CA = mp[SIMPLYP_P_CCOVER_A];
  if (dynamic_erod) {
    const double f_spr = sp[SIMPLYP_SC_F_SPR];
    CA = f_spr * season_cover(doy, mp[SIMPLYP_P_D_MAXE_SPR], CA)
         + (1.0 - f_spr) * season_cover(doy, mp[SIMPLYP_P_D_MAXE_AUT], CA);   // :579-580
  }
  aux.C_cover_A = CA;
  h.cM = c.m1 * CA + c.m2;                                       // :141-143
  // EPC0 (:600-611)
  double EPC0_A, EPC0_NC;
  if (dynamic_epc0) {
    const double iKM = sp_rcp(c.KfMsoil);
    EPC0_A = sp_max(c.PlabA * iKM, 0.0);
    EPC0_NC = sp_max(c.PlabNC * iKM, 0.0);
  } else {
    EPC0_A = mp[SIMPLYP_P_EPC0_A] * c.A_catch;
    EPC0_NC = fl.nc_is_S ? EPC0_A : mp[SIMPLYP_P_EPC0_S] * c.A_catch;
  }
  aux.EPC0_A = EPC0_A;
  aux.EPC0_NC = EPC0_NC;
  // TDP source coefficients with today's soil-water concentrations (:154-166)
  const double cTA = c.tdpA * c.concA;
  const double cTNC = c.tdpNC * c.concNC;
  const double omb = 1.0 - h.beta;
  if (fl.nc_is_A) { h.tA = omb * (cTA + cTNC); h.tS = 0.0; }
  else            { h.tA = omb * cTA;          h.tS = omb * cTNC; }
  h.t0 = (cTA + cTNC) * Qq + c.tdp_fixed + us[2];
  // PP source coefficient with today's labile P (:171-176)
  const double pA = c.PlabA + c.P_inactive, pN = c.PlabNC + c.P_inactive;
  h.cP = c.inv_Msoil_EPP * ((c.pp1 * CA + c.pp2) * pA + c.pp3 + (c.pp4 * CA + c.pp5) * pN);
}

// Post-ODE part of one day (:648-715).  Applies the groundwater floor to y, advances the soil-P
// carry in `c`, and fills the 13 non-ODE output values.
SP_HD void end_day(const Hot& h, Cold& c, const Flags& fl, int dynamic_epc0, const DayAux& aux,
                   double (&y)[NL], double (&non)[13]) {
  const double xA = y[iVsA] - h.fc, xS = y[iVsS] - h.fc;
  const double QsA = xA * gate(xA * h.inv_fcd) * h.inv_TsA;      // :663-664
  const double QsS = xS * gate(xS * h.inv_fcd) * h.inv_TsS;
  const double xg = y[iVg] * h.inv_Tg - h.Qg_min;                // :668-670
  const double Qg = h.Qg_min + gate(xg * h.inv_Qgd) * xg;
  y[iVg] = Qg * c.T_g;                                           // :670
  const double VsNC = fl.post_nc_is_A ? y[iVsA] : y[iVsS];       // :676-681
  const double QsNC = fl.post_nc_is_A ? QsA : QsS;
  if (dynamic_epc0) {                                            // :684-703
    soilp_update(c.pnetA, c.KfMsoil, aux.EPC0_A, QsA, aux.Qq, y[iVsA], c.TDPsA, c.PlabA);
    soilp_update(c.pnetNC, c.KfMsoil, aux.EPC0_NC, QsNC, aux.Qq, VsNC, c.TDPsNC, c.PlabNC);
    c.TDPsA = sp_max(c.TDPsA, 0.0);
    c.PlabA = sp_max(c.PlabA, 0.0);
    c.TDPsNC = sp_max(c.TDPsNC, 0.0);
    c.PlabNC = sp_max(c.PlabNC, 0.0);
    c.concA = c.TDPsA * sp_rcp(y[iVsA]);
    c.concNC = c.TDPsNC * sp_rcp(VsNC);
  } else {                                                       // :707-715
    c.concA = aux.EPC0_A;
    c.concNC = aux.EPC0_NC;
  }
  non[0] = aux.Qq;  non[1] = QsA;  non[2] = QsS;  non[3] = Qg;  non[4] = aux.C_cover_A;
  non[5] = aux.EPC0_A;  non[6] = aux.EPC0_NC;
  non[7] = c.TDPsA;  non[8] = c.PlabA;  non[9] = c.concA;
  non[10] = c.TDPsNC;  non[11] = c.PlabNC;  non[12] = c.concNC;
}

// ------------------------------------------------------------------------------------------
// Embedded explicit Runge-Kutta 5(4) with FSAL: Tsitouras' pair (-DSP_DOPRI5 selects Dormand-Prince).
namespace dp {
#ifndef SP_DOPRI5
// Tsitouras 5(4) (Ch. Tsitouras, Comput. Math. Appl. 62 (2011) 770-775): same 7-stage FSAL structure as
// Dormand-Prince but smaller principal error coefficients -> fewer steps at equal accuracy.
constexpr double a21 = 0.161;
constexpr double a31 = -0.008480655492356989, a32 = 0.335480655492357;
constexpr double a41 = 2.8971530571054935, a42 = -6.359448489975075, a43 = 4.3622954328695815;
constexpr double a51 = 5.325864828439257, a52 = -11.748883564062828, a53 = 7.4955393428898365, a54 = -0.09249506636175525;
constexpr double a61 = 5.86145544294642, a62 = -12.92096931784711, a63 = 8.159367898576159, a64 = -0.071584973281401,
                 a65 = -0.028269050394068383;
constexpr double b1 = 0.09646076681806523, b2 = 0.01, b3 = 0.4798896504144996, b4 = 1.379008574103742,
                 b5 = -3.290069515436081, b6 = 2.324710524099774;
constexpr double e1 = -0.00178001105222577714, e2 = -0.0008164344596567469, e3 = 0.007880878010261995,
                 e4 = -0.1447110071732629, e5 = 0.5823571654525552, e6 = -0.45808210592918697, e7 = 0.015151515151515152;
#else
// Dormand-Prince 5(4)
constexpr double a21 = 1.0 / 5.0;
constexpr double a31 = 3.0 / 40.0, a32 = 9.0 / 40.0;
constexpr double a41 = 44.0 / 45.0, a42 = -56.0 / 15.0, a43 = 32.0 / 9.0;
constexpr double a51 = 19372.0 / 6561.0, a52 = -25360.0 / 2187.0, a53 = 64448.0 / 6561.0, a54 = -212.0 / 729.0;
constexpr double a61 = 9017.0 / 3168.0, a62 = -355.0 / 33.0, a63 = 46732.0 / 5247.0, a64 = 49.0 / 176.0,
                 a65 = -5103.0 / 18656.0;
constexpr double b1 = 35.0 / 384.0, b2 = 0.0, b3 = 500.0 / 1113.0, b4 = 125.0 / 192.0, b5 = -2187.0 / 6784.0, b6 = 11.0 / 84.0;
constexpr double e1 = 71.0 / 57600.0, e2 = 0.0, e3 = -71.0 / 16695.0, e4 = 71.0 / 1920.0, e5 = -17253.0 / 339200.0,
                 e6 = 22.0 / 525.0, e7 = -1.0 / 40.0;
#endif
}  // namespace dp

// The same tableau as a constant-bank table: a DFMA/DMUL reads a c[bank][offset] operand directly, whereas a
// 64-bit literal is rematerialised with two moves at every use (the quad kernel has no registers to park 34
// constants in).
enum { RA21 = 0, RA31, RA32, RA41, RA42, RA43, RA51, RA52, RA53, RA54, RA61, RA62, RA63, RA64, RA65,
       RB1, RB2, RB3, RB4, RB5, RB6, RE1, RE2, RE3, RE4, RE5, RE6, RE7, RK_N };
SP_CONST double kRK[RK_N] = {
    dp::a21, dp::a31, dp::a32, dp::a41, dp::a42, dp::a43, dp::a51, dp::a52, dp::a53, dp::a54,
    dp::a61, dp::a62, dp::a63, dp::a64, dp::a65, dp::b1, dp::b2, dp::b3, dp::b4, dp::b5, dp::b6,
    dp::e1, dp::e2, dp::e3, dp::e4, dp::e5, dp::e6, dp::e7};

// The same controller on the MEAN SQUARE of the scaled error (no square root): 0.9*(en^2)^(-1/10) in [0.2, cap], cap <= 5
// (the caller passes 1 where the step must not grow: after a rejection and on the step after one).
// Device: fp32 lg2/ex2 with flush-to-zero and no range branches — an underflowing en^2 gives lg2 = -inf, hence
// +inf, clamped to cap; an overflowing one gives 0, and a NaN gives NaN, both clamped to 0.2 (fmaxf drops the NaN).
// `expo` = -1/(2p) for an estimate of order p-1 ... i.e. -0.1 for the 5(4) pair, -0.125 for Kaps-Rentrop 4(3).
#ifndef SP_CTRL_SAFETY
#define SP_CTRL_SAFETY 0.9     // scripts/controller_exp.py: 0.95 saves 2.8 % attempts at the price of 1.5x the rejections
#define SP_CTRL_MAXGROW 5.0
#endif
SP_HD double step_factor_sq(double en2, double expo = -0.1, double cap = SP_CTRL_MAXGROW) {
#if defined(__CUDA_ARCH__)
  float l, f;
  const float x = __double2float_rn(en2);
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(x));
  l *= (float)expo;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(f) : "f"(l));
  return (double)fminf(fmaxf((float)SP_CTRL_SAFETY * f, 0.2f), (float)cap);
#else
  if (en2 != en2) return 0.2;
  if (!(en2 > 1e-38)) return cap;
  if (!(en2 < 1e38)) return 0.2;
  const double f = SP_CTRL_SAFETY * exp(expo * log(en2));
  return sp_min(cap, sp_min(SP_CTRL_MAXGROW, sp_max(0.2, f)));
#endif
}

}  // namespace simplyp
