// simplyp_nsga2.cuh — per-pair and per-point arithmetic of NSGA-II (simplyp_nsga2_*_device, include/simplyp_b200.h).
//
// Deb et al. (2002), as the reference C code v1.1.6 runs it, with real variables in the unit cube (yl = 0, yu = 1);
// parameter values are de_scale's (simplyp_de.cuh).  Deviations from the reference code:
//   - selection: each parent is the better of two distinct members drawn uniformly, not the winner of Deb's two
//     permutation tournaments; "better" is lower rank, then larger crowding, then lower index (Deb breaks a full tie
//     with a coin);
//   - every draw is counter-based (below) rather than from one sequential generator, and a decision with probability
//     p is u < p with u in [0, 1) (Deb: u <= p), so p = 0 and p = 1 are exact;
//   - infeasible members (a status bit, or an objective that is not a finite number) dominate nothing and form the
//     last rank, ordered among themselves by index (crowding 0); Deb's constraint handling is not used;
//   - crowding breaks ties in an objective by index, sums the objectives in index order, and the survivors of the
//     last front are chosen by (crowding desc, index asc), so that the result is a function of the input only;
//   - ranking stops once at least N of the 2N points are ranked; the unranked points never survive.
//
// Random words: Philox4x32-10 (simplyp_mcmc.cuh) keyed by the 64-bit seed.  Pair p at generation g takes its group q of
// four words from counter (p, g lo, g hi, 5 + 256 q):
//   group 0:          tournament picks a = mulhi(w0, N), b = mulhi(w1, N - 1) shifted past a; c, d likewise from
//                     w2, w3 (parent 1 = better of a, b; parent 2 = better of c, d);
//   group 1:          u53(w0, w1): SBX on the pair when < crossover (w2, w3 unused);
//   group 2 + 4j:     u53(w0, w1): variable j crosses when < 0.5;  u53(w2, w3): the SBX random number of variable j;
//   group 3 + 4j:     u53(w0, w1): the two children of variable j are swapped when < 0.5 (w2, w3 unused);
//   group 4 + 4j:     child 1: u53(w0, w1) mutates variable j when < mutation;  u53(w2, w3): its random number;
//   group 5 + 4j:     child 2, the same.
// The last counter word is 5 modulo 256, so no NSGA-II draw collides with the sampler's blocks 0 and 1, the bands'
// block 2, the Sobol' bootstrap's block 3 or differential evolution's block 4.  Every draw is a function of (seed,
// pair, generation) only, so a run does not depend on launch geometry and a continued run draws what a longer one
// would.
//
// Arithmetic: every operation is rounded on its own (mc_add / mc_sub / mc_mul / mc_div), so nvcc cannot contract
// anything into an FMA.  The exceptions are the pow calls of SBX and of polynomial mutation: the device's pow and the
// host's libm can differ in the last bits, so offspring agree with a NumPy restatement to a stated ulp bound
// (tests/test_nsga2_cpu.py) and every discrete decision agrees exactly.  Ranks, crowding and survivors use comparisons
// and mc_* operations only and agree bit for bit.
//
// Inline __host__ __device__ code like simplyp_de.cuh: the CPU test tier compiles it for the host.
#pragma once

#include "simplyp_de.cuh"

namespace simplyp {

constexpr uint32_t NSGA2_BLOCK = 5;   // counter word 3 of group q is NSGA2_BLOCK + 256 q
constexpr double NSGA2_EPS = 1e-14;   // SBX leaves a variable alone when |x1 - x2| <= EPS (Deb's EPS)

SP_HD void nsga2_words(uint64_t seed, long long g, uint32_t pair, int group, uint32_t (&r)[4]) {
  const uint64_t ug = (uint64_t)g;
  const uint32_t ctr[4] = {pair, (uint32_t)ug, (uint32_t)(ug >> 32), NSGA2_BLOCK + 256u * (uint32_t)group};
  philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32), r);
}

// The better of members a and b: lower rank, then larger crowding, then lower index.
SP_HD int nsga2_better(const int32_t* rank, const double* crowd, int a, int b) {
  if (rank[a] != rank[b]) return rank[a] < rank[b] ? a : b;
  if (crowd[a] != crowd[b]) return crowd[a] > crowd[b] ? a : b;
  return a < b ? a : b;
}

// Tournament picks of pair p at generation g: picks[4] = a, b, c, d (a != b, c != d).
SP_HD void nsga2_picks(const SimplypNsga2& ns, long long g, int p, int (&picks)[4]) {
  const uint32_t N = (uint32_t)ns.n_population;
  uint32_t w[4];
  nsga2_words(ns.seed, g, (uint32_t)p, 0, w);
  for (int t = 0; t < 2; ++t) {
    const int a = (int)mc_mulhi(w[2 * t], N);
    int b = (int)mc_mulhi(w[2 * t + 1], N - 1);
    b += b >= a;
    picks[2 * t] = a;
    picks[2 * t + 1] = b;
  }
}

// SBX's spread factor beta_q for the bound distance term `beta` (Deb's realcross, one side).
SP_HD double nsga2_betaq(double beta, double rand, double eta_c) {
  const double expo = mc_add(eta_c, 1.0);
  const double alpha = mc_sub(2.0, pow(beta, -expo));
  if (rand <= mc_div(1.0, alpha)) return pow(mc_mul(rand, alpha), mc_div(1.0, expo));
  return pow(mc_div(1.0, mc_sub(2.0, mc_mul(rand, alpha))), mc_div(1.0, expo));
}

// Polynomial mutation of y in [0, 1] with random number rnd (Deb's real_mutate_ind, yl = 0, yu = 1: delta1 = y,
// delta2 = 1 - y, and the step deltaq (yu - yl) = deltaq), clamped to [0, 1].
SP_HD double nsga2_mutate(double y, double rnd, double eta_m) {
  const double expo = mc_add(eta_m, 1.0), mut_pow = mc_div(1.0, expo);
  double deltaq;
  if (rnd <= 0.5) {
    const double xy = mc_sub(1.0, y);
    const double val = mc_add(mc_mul(2.0, rnd), mc_mul(mc_sub(1.0, mc_mul(2.0, rnd)), pow(xy, expo)));
    deltaq = mc_sub(pow(val, mut_pow), 1.0);
  } else {
    const double xy = mc_sub(1.0, mc_sub(1.0, y));
    const double val = mc_add(mc_mul(2.0, mc_sub(1.0, rnd)), mc_mul(mc_mul(2.0, mc_sub(rnd, 0.5)), pow(xy, expo)));
    deltaq = mc_sub(1.0, pow(val, mut_pow));
  }
  const double v = mc_add(y, deltaq);
  return v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
}

// Decision bits of one variable, for the tests: SBX applied, children swapped, child 1 / child 2 mutated.
enum { NSGA2_D_SBX = 1, NSGA2_D_SWAP = 2, NSGA2_D_MUT1 = 4, NSGA2_D_MUT2 = 8 };

// Offspring pair p at generation g from the population pop[N][K] with rank[N] and crowd[N]: children c1[K], c2[K].
// dec (may be NULL): [3 + K] = parent 1, parent 2, pair crossed, then the decision bits of every variable.
SP_HD void nsga2_offspring_pair(const SimplypNsga2& ns, const double* pop, const int32_t* rank, const double* crowd,
                                long long g, int p, double* c1, double* c2, int32_t* dec) {
  const int K = ns.n_free;
  int picks[4];
  nsga2_picks(ns, g, p, picks);
  const int p1 = nsga2_better(rank, crowd, picks[0], picks[1]);
  const int p2 = nsga2_better(rank, crowd, picks[2], picks[3]);
  const double* x1 = pop + (size_t)p1 * K;
  const double* x2 = pop + (size_t)p2 * K;
  uint32_t w[4];
  nsga2_words(ns.seed, g, (uint32_t)p, 1, w);
  const int cross = mcmc_u53(w[0], w[1]) < ns.crossover;
  if (dec) { dec[0] = p1; dec[1] = p2; dec[2] = cross; }
  for (int j = 0; j < K; ++j) {
    int bits = 0;
    double a = x1[j], b = x2[j];
    if (cross) {
      nsga2_words(ns.seed, g, (uint32_t)p, 2 + 4 * j, w);
      const double rand = mcmc_u53(w[2], w[3]);
      if (mcmc_u53(w[0], w[1]) < 0.5 && fabs(mc_sub(a, b)) > NSGA2_EPS) {
        const double y1 = a < b ? a : b, y2 = a < b ? b : a, d = mc_sub(y2, y1);
        double bq = nsga2_betaq(mc_add(1.0, mc_div(mc_mul(2.0, y1), d)), rand, ns.eta_c);
        double v1 = mc_mul(0.5, mc_sub(mc_add(y1, y2), mc_mul(bq, d)));
        bq = nsga2_betaq(mc_add(1.0, mc_div(mc_mul(2.0, mc_sub(1.0, y2)), d)), rand, ns.eta_c);
        double v2 = mc_mul(0.5, mc_add(mc_add(y1, y2), mc_mul(bq, d)));
        v1 = v1 < 0.0 ? 0.0 : (v1 > 1.0 ? 1.0 : v1);
        v2 = v2 < 0.0 ? 0.0 : (v2 > 1.0 ? 1.0 : v2);
        nsga2_words(ns.seed, g, (uint32_t)p, 3 + 4 * j, w);
        const int swap = mcmc_u53(w[0], w[1]) < 0.5;
        a = swap ? v2 : v1;
        b = swap ? v1 : v2;
        bits |= NSGA2_D_SBX | (swap ? NSGA2_D_SWAP : 0);
      }
    }
    nsga2_words(ns.seed, g, (uint32_t)p, 4 + 4 * j, w);
    if (mcmc_u53(w[0], w[1]) < ns.mutation) { a = nsga2_mutate(a, mcmc_u53(w[2], w[3]), ns.eta_m); bits |= NSGA2_D_MUT1; }
    nsga2_words(ns.seed, g, (uint32_t)p, 5 + 4 * j, w);
    if (mcmc_u53(w[0], w[1]) < ns.mutation) { b = nsga2_mutate(b, mcmc_u53(w[2], w[3]), ns.eta_m); bits |= NSGA2_D_MUT2; }
    c1[j] = a;
    c2[j] = b;
    if (dec) dec[3 + j] = bits;
  }
}

// Oriented objectives f[M] of a member from its values y (y[m * stride]) and its status: NaN everywhere when the
// status is set or a value is not finite.  Returns 1 when feasible.
SP_HD int nsga2_orient(const SimplypNsga2& ns, const double* y, long long stride, int status, double* f) {
  const int M = ns.n_objectives;
  int ok = !status;
  for (int m = 0; m < M; ++m) {
    const double v = y[(size_t)m * stride];
    ok &= fabs(v) < INFINITY;
  }
  for (int m = 0; m < M; ++m) f[m] = ok ? mc_mul(ns.sense[m], y[(size_t)m * stride]) : NAN;
  return ok;
}

// Whether fa dominates fb (oriented, larger is better): fa >= fb everywhere and fa > fb somewhere.  A NaN row (an
// infeasible point) neither dominates nor is dominated.
// The loop runs to the compile-time bound so that fb may be an array the caller holds in registers.
SP_HD int nsga2_dominates(const double* fa, const double* fb, int M) {
  int ge = 1, gt = 0;
#pragma unroll
  for (int m = 0; m < SIMPLYP_NSGA2_MAX_OBJECTIVES; ++m) {
    if (m < M) {
      ge &= fa[m] >= fb[m];
      gt |= fa[m] > fb[m];
    }
  }
  return ge & gt;
}

// Crowding term of one objective: +inf at either end of the front's order, 0 for a constant objective, else
// (next - prev) / (max - min).
SP_HD double nsga2_crowd_term(int boundary, double next, double prev, double mx, double mn) {
  if (boundary) return INFINITY;
  if (mx == mn) return 0.0;
  return mc_div(mc_sub(next, prev), mc_sub(mx, mn));
}

}  // namespace simplyp
