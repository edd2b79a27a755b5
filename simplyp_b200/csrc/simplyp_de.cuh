// simplyp_de.cuh — per-member arithmetic of differential evolution (simplyp_de_*_device, include/simplyp_b200.h).
//
// scipy.optimize.differential_evolution with updating='deferred' (synchronous generations), strategies best1bin and
// rand1bin, binomial crossover, no polishing.  The population lives in the unit cube [0, 1]^K as scipy's does; a
// parameter value is arg1 + (u - 0.5) arg2, arg1 = 0.5 (lo + hi), arg2 = |hi - lo| (scipy's _scale_parameters), and
// is then clamped to [lo, hi] so that a last-bit rounding never hands the integrator an out-of-box value.  The clamp
// is the only intended deviation from scipy's arithmetic.  Every operation is rounded on its own (mc_add / mc_sub /
// mc_mul), so nvcc cannot contract anything into an FMA and a NumPy restatement matches bit for bit.
//
// Trial of member i at generation g (F the generation's mutation factor, x the population, b the best member):
//   best1bin: b'_j = x_b,j + F (x_r0,j - x_r1,j);   rand1bin: b'_j = x_r0,j + F (x_r1,j - x_r2,j)
//   t_j = b'_j if u_j < CR or j == fill, else x_i,j;   a t_j outside [0, 1] is replaced by a fresh uniform v_j
//   (scipy's _ensure_constraint).
// Random words: Philox4x32-10 (simplyp_mcmc.cuh) keyed by the 64-bit seed.  Member i at generation g takes its group
// q of four words from counter (i, g lo, g hi, 4 + 256 q):
//   group 0: r0 = mulhi(w0, N - 1), r1 = mulhi(w1, N - 2), r2 = mulhi(w2, N - 3) (rand1bin only), fill = mulhi(w3, K);
//            each pick is shifted past the indices already taken (i, then r0, then r1, in ascending order), so the
//            picks are distinct, differ from i and are uniform without a rejection loop;
//   group 1 + j: u_j = u53(w0, w1) (crossover), v_j = u53(w2, w3) (redraw).
// The mutation factor F = lo + (hi - lo) u53(w0, w1) is drawn once per generation (scipy's dither) from counter
// (0xFFFFFFFF, g lo, g hi, 4).  The last counter word is 4 modulo 256, so no DE draw collides with the sampler's
// blocks 0 and 1, the bands' block 2 or the Sobol' bootstrap's block 3.  Every draw is a function of (seed, member,
// generation) only, so a run does not depend on launch geometry and a continued run draws what a longer one would.
//
// Selection (scipy's _accept_trial without constraints): the trial replaces its target when E_trial <= E_target.
// E = -sum_r w_r y_r over the objective rows y of the member; a non-zero status word of the member's integration, or a
// sum that is not a number, gives E = +inf.
//
// Inline __host__ __device__ code like simplyp_mcmc.cuh: the CPU test tier compiles it for the host.
#pragma once

#include "simplyp_mcmc.cuh"

namespace simplyp {

constexpr uint32_t DE_BLOCK = 4;                  // counter word 3 of group q is DE_BLOCK + 256 q
constexpr uint32_t DE_DITHER_MEMBER = 0xFFFFFFFFu;

SP_HD void de_words(uint64_t seed, long long g, uint32_t member, int group, uint32_t (&r)[4]) {
  const uint64_t ug = (uint64_t)g;
  const uint32_t ctr[4] = {member, (uint32_t)ug, (uint32_t)(ug >> 32), DE_BLOCK + 256u * (uint32_t)group};
  philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32), r);
}

// The mutation factor of generation g.
SP_HD double de_dither(const SimplypDe& de, long long g) {
  uint32_t r[4];
  de_words(de.seed, g, DE_DITHER_MEMBER, 0, r);
  return mc_add(de.mutation_lo, mc_mul(mc_sub(de.mutation_hi, de.mutation_lo), mcmc_u53(r[0], r[1])));
}

// Picks r[0..n_picks) of member i (n_picks = 2 for best1bin, 3 for rand1bin) and the fill point.
SP_HD void de_picks(const SimplypDe& de, long long g, int i, int (&r)[3], int* fill) {
  const int N = de.n_population, n_picks = de.strategy == SIMPLYP_DE_RAND1BIN ? 3 : 2;
  uint32_t w[4];
  de_words(de.seed, g, (uint32_t)i, 0, w);
  int taken[4] = {i, 0, 0, 0};   // ascending
  for (int p = 0; p < n_picks; ++p) {
    int v = (int)mc_mulhi(w[p], (uint32_t)(N - 1 - p));
    for (int q = 0; q <= p; ++q) v += v >= taken[q];
    r[p] = v;
    int q = p + 1;
    for (; q > 0 && taken[q - 1] > v; --q) taken[q] = taken[q - 1];
    taken[q] = v;
  }
  if (n_picks == 2) r[2] = -1;
  *fill = (int)mc_mulhi(w[3], (uint32_t)de.n_free);
}

// Trial trial[K] of member i at generation g from the population pop[N][K] with best member `best`.
SP_HD void de_trial_member(const SimplypDe& de, const double* pop, long long best, long long g, int i, double F,
                           double* trial) {
  const int K = de.n_free;
  int r[3], fill;
  de_picks(de, g, i, r, &fill);
  const int rand1 = de.strategy == SIMPLYP_DE_RAND1BIN;
  const double* xa = pop + (size_t)(rand1 ? r[0] : best) * K;
  const double* xb = pop + (size_t)(rand1 ? r[1] : r[0]) * K;
  const double* xc = pop + (size_t)(rand1 ? r[2] : r[1]) * K;
  const double* xi = pop + (size_t)i * K;
  for (int j = 0; j < K; ++j) {
    uint32_t w[4];
    de_words(de.seed, g, (uint32_t)i, 1 + j, w);
    double t = xi[j];
    if (mcmc_u53(w[0], w[1]) < de.recombination || j == fill) t = mc_add(xa[j], mc_mul(F, mc_sub(xb[j], xc[j])));
    if (t > 1.0 || t < 0.0) t = mcmc_u53(w[2], w[3]);
    trial[j] = t;
  }
}

// Parameter value of unit-cube coordinate u in the box of p, clamped to [lo, hi].
SP_HD double de_scale(const SimplypMcmcParam& p, double u) {
  const double arg1 = mc_mul(0.5, mc_add(p.lo, p.hi)), arg2 = fabs(mc_sub(p.lo, p.hi));
  const double v = mc_add(arg1, mc_mul(mc_sub(u, 0.5), arg2));
  return v < p.lo ? p.lo : (v > p.hi ? p.hi : v);
}

// Energy of member m from the objective rows y[R][N] (weights w[R]) and its status words diag[S][SIMPLYP_NDIAG].
SP_HD double de_energy(const double* y, long long N, int R, const double* w, long long m, const int64_t* diag,
                       int S) {
  for (int s = 0; s < S; ++s)
    if (diag[(size_t)s * SIMPLYP_NDIAG + SIMPLYP_DG_STATUS] != 0) return INFINITY;
  double acc = 0.0;
  for (int r = 0; r < R; ++r) acc = mc_add(acc, mc_mul(w[r], y[(size_t)r * N + m]));
  const double e = -acc;
  return e < INFINITY ? e : INFINITY;   // NaN and +inf -> +inf
}

// Selection of member i: the trial replaces its target when e_trial <= energy[i].  Returns 1 on replacement.
SP_HD int de_select_member(int K, int i, double e_trial, const double* trial, double* pop, double* energy) {
  if (!(e_trial <= energy[i])) return 0;
  for (int j = 0; j < K; ++j) pop[(size_t)i * K + j] = trial[j];
  energy[i] = e_trial;
  return 1;
}

}  // namespace simplyp
