// simplyp_morris.cuh — arithmetic of the Morris elementary-effects screening (simplyp_morris_*_device,
// include/simplyp_b200.h).
//
// Levels.  K free parameters, p = num_levels (even, 2..16), h = p / 2 and Delta = p / (2 (p - 1)).  A point of a
// trajectory is a vector of integer levels 0..p-1; level l has the unit value u = l / (p - 1) (one rounded division)
// and the parameter value min(lo + (hi - lo) u, hi), each operation rounded on its own, as in the Sobol' design.
//
// Candidate trajectory c: a base level b_z in 0..h-1, a direction d_z = +-1 and a step order pi (a permutation of the
// K coordinates).  Point 0 puts z at b_z (d_z = +1) or b_z + h (d_z = -1); step s = 1..K moves coordinate pi(s-1) by
// d h levels, which is Delta in the unit cube, so every coordinate moves exactly once.  This is Morris' (1991)
// B* = (J x* + Delta/2 ((2B - J) D* + J)) P* in levels.  Stored form (4 K bytes a candidate, morris_traj_pack):
//   x0[z]  level of z at point 0;   pos[z] the step that moves z, minus 1;   ord[s] = pi(s);   neg[z] = 1 if d_z = -1.
//
// Random words: Philox4x32-10 keyed by the seed.  Word k of candidate c is word k mod 4 of the block with counter
// (c, k / 4, 0, 6); integer picks in 0..n-1 are (w n) >> 32, as the Sobol' bootstrap takes them:
//   words 0 .. K-1         b_z = pick(w_z, h)
//   words K .. 2K-1        d_z = -1 if pick(w_{K+z}, 2) = 1 (the top bit of the word), else +1
//   words 2K .. 3K-2       Fisher-Yates from pi = identity: for i = K-1 down to 1, word 2K + (K-1-i) picks
//                          j = pick(w, i + 1) and swaps pi(i) and pi(j)
// Bootstrap resample b draws n of a row's used trajectories with replacement; draw k picks used position (w n) >> 32,
// w = word k mod 4 of the block with counter (b, k / 4, 1, 6).  Block 6 is disjoint from the sampler's blocks 0 and 1
// (simplyp_mcmc.cuh), the bands' block 2, the Sobol' bootstrap's block 3, DE's 4 + 256 q and NSGA-II's 5 + 256 q.
//
// Optimised trajectories (Campolongo et al. 2007) by the greedy search of Ruano et al. (2012), NOT SALib's exact
// routine: the distance of candidates m < l is
//   d(m, l) = sum over i = 0..K, then j = 0..K, of sqrt(sum_z (L_m[i][z] - L_l[j][z])^2)
// in level units: each inner sum an exact integer, each sqrt correctly rounded, the outer sum one running total in
// that order (i-major), one rounding per addition; d(l, m) is d(m, l), always formed with the lower index first.  The
// selection starts from the pair with the largest d (ties: the lowest (m, l)), then repeatedly adds the candidate c
// that maximises sum over the selected s, in the order they were selected, of d(c, s)^2 (ties: the lowest c).
//
// Inline __host__ __device__ code like simplyp_sobol.cuh: the CPU test tier compiles it for the host.
#pragma once

#include "simplyp_mcmc.cuh"

namespace simplyp {

constexpr uint32_t MORRIS_BLOCK = 6;     // the fourth counter word of every Morris draw

// Philox word k of candidate (or resample) a; third counter word `kind` (0: trajectory, 1: bootstrap).
SP_HD void morris_words(uint64_t seed, uint32_t a, uint32_t q, uint32_t kind, uint32_t (&r)[4]) {
  const uint32_t ctr[4] = {a, q, kind, MORRIS_BLOCK};
  philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32), r);
}

SP_HD uint32_t morris_pick(uint32_t w, uint32_t n) { return (uint32_t)(((uint64_t)w * n) >> 32); }

// Candidate c in stored form: t[0..K) x0, t[K..2K) pos, t[2K..3K) ord, t[3K..4K) neg.
SP_HD void morris_traj_pack(uint64_t seed, uint32_t c, int K, int p, uint8_t* t) {
  const uint32_t h = (uint32_t)(p / 2);
  uint8_t* x0 = t;
  uint8_t* pos = t + K;
  uint8_t* ord = t + 2 * K;
  uint8_t* neg = t + 3 * K;
  for (int z = 0; z < K; ++z) ord[z] = (uint8_t)z;
  uint32_t r[4];
  const int n_words = 3 * K - 1;
  for (int k = 0; k < n_words; ++k) {
    if ((k & 3) == 0) morris_words(seed, c, (uint32_t)(k >> 2), 0u, r);
    const uint32_t w = r[k & 3];
    if (k < K) {
      x0[k] = (uint8_t)morris_pick(w, h);
    } else if (k < 2 * K) {
      neg[k - K] = (uint8_t)morris_pick(w, 2);
    } else {
      const int i = K - 1 - (k - 2 * K);
      const int j = (int)morris_pick(w, (uint32_t)(i + 1));
      const uint8_t tmp = ord[i];
      ord[i] = ord[j];
      ord[j] = tmp;
    }
  }
  for (int z = 0; z < K; ++z) {
    if (neg[z]) x0[z] = (uint8_t)(x0[z] + h);
    pos[ord[z]] = (uint8_t)z;
  }
}

// Signed move of coordinate z (+h or -h levels).
SP_HD int morris_move(const uint8_t* t, int K, int h, int z) { return t[3 * K + z] ? -h : h; }

// Level of coordinate z at point s (0..K) of a stored trajectory.
SP_HD int morris_level(const uint8_t* t, int K, int h, int s, int z) {
  return t[z] + (t[K + z] < s ? morris_move(t, K, h, z) : 0);
}

SP_HD double morris_unit(int level, int p) { return mc_div((double)level, (double)(p - 1)); }

// lo + (hi - lo) u can round above hi at the top level: the value is clamped to the box.
SP_HD double morris_value(const SimplypMcmcParam& q, int level, int p) {
  const double v = mc_add(q.lo, mc_mul(mc_sub(q.hi, q.lo), morris_unit(level, p)));
  return v < q.hi ? v : q.hi;
}

SP_HD double morris_delta(int p) { return mc_div((double)p, (double)(2 * (p - 1))); }

SP_HD double morris_sqrt(int q) {
#if defined(__CUDA_ARCH__)
  return __dsqrt_rn((double)q);
#else
  return std::sqrt((double)q);
#endif
}

// d(a, b) of two stored trajectories (a the lower candidate index).  The squared distance of point pair (i, j) is
// carried exactly from its neighbour: moving from point i-1 to i of a (or j-1 to j of b) changes one coordinate.
SP_HD double morris_distance(const uint8_t* a, const uint8_t* b, int K, int h) {
  int d0 = 0;
  for (int z = 0; z < K; ++z) {
    const int e = (int)a[z] - (int)b[z];
    d0 += e * e;
  }
  double total = 0.0;
  for (int i = 0; i <= K; ++i) {
    if (i > 0) {
      const int z = a[2 * K + i - 1], ao = a[z], an = ao + morris_move(a, K, h, z), bv = b[z];
      d0 += (an - bv) * (an - bv) - (ao - bv) * (ao - bv);
    }
    int d = d0;
    for (int j = 0; j <= K; ++j) {
      if (j > 0) {
        const int z = b[2 * K + j - 1], av = morris_level(a, K, h, i, z), bo = b[z],
                  bn = bo + morris_move(b, K, h, z);
        d += (av - bn) * (av - bn) - (av - bo) * (av - bo);
      }
      total = mc_add(total, morris_sqrt(d));
    }
  }
  return total;
}

}  // namespace simplyp
