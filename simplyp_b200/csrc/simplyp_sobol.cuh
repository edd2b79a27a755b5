// simplyp_sobol.cuh — arithmetic of the Sobol' sensitivity analysis (simplyp_sobol_*_device, include/simplyp_b200.h).
//
// Design: unscrambled Sobol' points in 2K dimensions with the Joe-Kuo direction numbers (new-joe-kuo-6.21201, the
// table SciPy's qmc.Sobol ships).  Point n is the XOR, over the set bits j of gray(n) = n ^ (n >> 1), of the 32-bit
// direction numbers V[d][j], and u = x 2^-32: every point is computed on its own, so one thread writes one member.
// The Saltelli design in SALib's row order: member m = i P + slot of sample i (Sobol' point skip + i) is A (slot 0,
// the point's first K coordinates), AB_j (slot 1 + j: A with column j from B, B being the last K coordinates),
// BA_j (slot K + 1 + j, second order only: B with column j from A) or B (slot P - 1); P = K + 2 or 2K + 2.
// A parameter value is lo + (hi - lo) u, every operation rounded on its own, so NumPy reproduces it bit for bit.
//
// Bootstrap: resample t draws n of the row's used samples with replacement; draw k picks used position
// (w n) >> 32, w = word k mod 4 of the Philox4x32-10 block keyed by the seed with counter (t, k / 4, 0, 3).  Block 3
// is disjoint from the sampler's blocks 0 and 1 (simplyp_mcmc.cuh) and the bands' block 2 (simplyp_bands.cuh).
//
// Inline __host__ __device__ code like simplyp_mcmc.cuh: the CPU test tier compiles it for the host.
#pragma once

#include "simplyp_mcmc.cuh"

namespace simplyp {

constexpr int SOBOL_DIMS = 2 * SIMPLYP_MCMC_MAX_FREE;   // 128: every polynomial of degree <= 10
constexpr int SOBOL_BITS = 32;
constexpr uint32_t SOBOL_BLOCK = 3;                     // the fourth counter word of the bootstrap draws

// Primitive polynomial (with its leading and trailing bits) and initial direction numbers m_1 .. m_deg of each
// dimension: the first 128 rows of SciPy's _sobol_direction_numbers.npz (dimension 0 is the van der Corput sequence).
struct SobolInit {
  uint32_t poly;
  uint32_t m[10];
};
constexpr SobolInit SOBOL_INIT[SOBOL_DIMS] = {
    {1, {1}}, {3, {1}}, {7, {1, 3}}, {11, {1, 3, 1}}, {13, {1, 1, 1}}, {19, {1, 1, 3, 3}}, {25, {1, 3, 5, 13}},
    {37, {1, 1, 5, 5, 17}}, {41, {1, 1, 5, 5, 5}}, {47, {1, 1, 7, 11, 19}}, {55, {1, 1, 5, 1, 1}},
    {59, {1, 1, 1, 3, 11}}, {61, {1, 3, 5, 5, 31}}, {67, {1, 3, 3, 9, 7, 49}}, {91, {1, 1, 1, 15, 21, 21}},
    {97, {1, 3, 1, 13, 27, 49}}, {103, {1, 1, 1, 15, 7, 5}}, {109, {1, 3, 1, 15, 13, 25}},
    {115, {1, 1, 5, 5, 19, 61}}, {131, {1, 3, 7, 11, 23, 15, 103}}, {137, {1, 3, 7, 13, 13, 15, 69}},
    {143, {1, 1, 3, 13, 7, 35, 63}}, {145, {1, 3, 5, 9, 1, 25, 53}}, {157, {1, 3, 1, 13, 9, 35, 107}},
    {167, {1, 3, 1, 5, 27, 61, 31}}, {171, {1, 1, 5, 11, 19, 41, 61}}, {185, {1, 3, 5, 3, 3, 13, 69}},
    {191, {1, 1, 7, 13, 1, 19, 1}}, {193, {1, 3, 7, 5, 13, 19, 59}}, {203, {1, 1, 3, 9, 25, 29, 41}},
    {211, {1, 3, 5, 13, 23, 1, 55}}, {213, {1, 3, 7, 3, 13, 59, 17}}, {229, {1, 3, 1, 3, 5, 53, 69}},
    {239, {1, 1, 5, 5, 23, 33, 13}}, {241, {1, 1, 7, 7, 1, 61, 123}}, {247, {1, 1, 7, 9, 13, 61, 49}},
    {253, {1, 3, 3, 5, 3, 55, 33}}, {285, {1, 3, 1, 15, 31, 13, 49, 245}}, {299, {1, 3, 5, 15, 31, 59, 63, 97}},
    {301, {1, 3, 1, 11, 11, 11, 77, 249}}, {333, {1, 3, 1, 11, 27, 43, 71, 9}}, {351, {1, 1, 7, 15, 21, 11, 81, 45}},
    {355, {1, 3, 7, 3, 25, 31, 65, 79}}, {357, {1, 3, 1, 1, 19, 11, 3, 205}}, {361, {1, 1, 5, 9, 19, 21, 29, 157}},
    {369, {1, 3, 7, 11, 1, 33, 89, 185}}, {391, {1, 3, 3, 3, 15, 9, 79, 71}}, {397, {1, 3, 7, 11, 15, 39, 119, 27}},
    {425, {1, 1, 3, 1, 11, 31, 97, 225}}, {451, {1, 1, 1, 3, 23, 43, 57, 177}}, {463, {1, 3, 7, 7, 17, 17, 37, 71}},
    {487, {1, 3, 1, 5, 27, 63, 123, 213}}, {501, {1, 1, 3, 5, 11, 43, 53, 133}},
    {529, {1, 3, 5, 5, 29, 17, 47, 173, 479}}, {539, {1, 3, 3, 11, 3, 1, 109, 9, 69}},
    {545, {1, 1, 1, 5, 17, 39, 23, 5, 343}}, {557, {1, 3, 1, 5, 25, 15, 31, 103, 499}},
    {563, {1, 1, 1, 11, 11, 17, 63, 105, 183}}, {601, {1, 1, 5, 11, 9, 29, 97, 231, 363}},
    {607, {1, 1, 5, 15, 19, 45, 41, 7, 383}}, {617, {1, 3, 7, 7, 31, 19, 83, 137, 221}},
    {623, {1, 1, 1, 3, 23, 15, 111, 223, 83}}, {631, {1, 1, 5, 13, 31, 15, 55, 25, 161}},
    {637, {1, 1, 3, 13, 25, 47, 39, 87, 257}}, {647, {1, 1, 1, 11, 21, 53, 125, 249, 293}},
    {661, {1, 1, 7, 11, 11, 7, 57, 79, 323}}, {675, {1, 1, 5, 5, 17, 13, 81, 3, 131}},
    {677, {1, 1, 7, 13, 23, 7, 65, 251, 475}}, {687, {1, 3, 5, 1, 9, 43, 3, 149, 11}},
    {695, {1, 1, 3, 13, 31, 13, 13, 255, 487}}, {701, {1, 3, 3, 1, 5, 63, 89, 91, 127}},
    {719, {1, 1, 3, 3, 1, 19, 123, 127, 237}}, {721, {1, 1, 5, 7, 23, 31, 37, 243, 289}},
    {731, {1, 1, 5, 11, 17, 53, 117, 183, 491}}, {757, {1, 1, 1, 5, 1, 13, 13, 209, 345}},
    {761, {1, 1, 3, 15, 1, 57, 115, 7, 33}}, {787, {1, 3, 1, 11, 7, 43, 81, 207, 175}},
    {789, {1, 3, 1, 1, 15, 27, 63, 255, 49}}, {799, {1, 3, 5, 3, 27, 61, 105, 171, 305}},
    {803, {1, 1, 5, 3, 1, 3, 57, 249, 149}}, {817, {1, 1, 3, 5, 5, 57, 15, 13, 159}},
    {827, {1, 1, 1, 11, 7, 11, 105, 141, 225}}, {847, {1, 3, 3, 5, 27, 59, 121, 101, 271}},
    {859, {1, 3, 5, 9, 11, 49, 51, 59, 115}}, {865, {1, 1, 7, 1, 23, 45, 125, 71, 419}},
    {875, {1, 1, 3, 5, 23, 5, 105, 109, 75}}, {877, {1, 1, 7, 15, 7, 11, 67, 121, 453}},
    {883, {1, 3, 7, 3, 9, 13, 31, 27, 449}}, {895, {1, 3, 1, 15, 19, 39, 39, 89, 15}},
    {901, {1, 1, 1, 1, 1, 33, 73, 145, 379}}, {911, {1, 3, 1, 15, 15, 43, 29, 13, 483}},
    {949, {1, 1, 7, 3, 19, 27, 85, 131, 431}}, {953, {1, 3, 3, 3, 5, 35, 23, 195, 349}},
    {967, {1, 3, 3, 7, 9, 27, 39, 59, 297}}, {971, {1, 1, 3, 9, 11, 17, 13, 241, 157}},
    {973, {1, 3, 7, 15, 25, 57, 33, 189, 213}}, {981, {1, 1, 7, 1, 9, 55, 73, 83, 217}},
    {985, {1, 3, 3, 13, 19, 27, 23, 113, 249}}, {995, {1, 3, 5, 3, 23, 43, 3, 253, 479}},
    {1001, {1, 1, 5, 5, 11, 5, 45, 117, 217}}, {1019, {1, 3, 3, 7, 29, 37, 33, 123, 147}},
    {1033, {1, 3, 1, 15, 5, 5, 37, 227, 223, 459}}, {1051, {1, 1, 7, 5, 5, 39, 63, 255, 135, 487}},
    {1063, {1, 3, 1, 7, 9, 7, 87, 249, 217, 599}}, {1069, {1, 1, 3, 13, 9, 47, 7, 225, 363, 247}},
    {1125, {1, 3, 7, 13, 19, 13, 9, 67, 9, 737}}, {1135, {1, 3, 5, 5, 19, 59, 7, 41, 319, 677}},
    {1153, {1, 1, 5, 3, 31, 63, 15, 43, 207, 789}}, {1163, {1, 1, 7, 9, 13, 39, 3, 47, 497, 169}},
    {1221, {1, 3, 1, 7, 21, 17, 97, 19, 415, 905}}, {1239, {1, 3, 7, 1, 3, 31, 71, 111, 165, 127}},
    {1255, {1, 1, 5, 11, 1, 61, 83, 119, 203, 847}}, {1267, {1, 3, 3, 13, 9, 61, 19, 97, 47, 35}},
    {1279, {1, 1, 7, 7, 15, 29, 63, 95, 417, 469}}, {1293, {1, 3, 1, 9, 25, 9, 71, 57, 213, 385}},
    {1305, {1, 3, 5, 13, 31, 47, 101, 57, 39, 341}}, {1315, {1, 1, 3, 3, 31, 57, 125, 173, 365, 551}},
    {1329, {1, 3, 7, 1, 13, 57, 67, 157, 451, 707}}, {1341, {1, 1, 1, 7, 21, 13, 105, 89, 429, 965}},
    {1347, {1, 1, 5, 9, 17, 51, 45, 119, 157, 141}}, {1367, {1, 3, 7, 7, 13, 45, 91, 9, 129, 741}},
    {1387, {1, 3, 7, 1, 23, 57, 67, 141, 151, 571}}, {1413, {1, 1, 3, 11, 17, 47, 93, 107, 375, 157}},
    {1423, {1, 3, 3, 5, 11, 21, 43, 51, 169, 915}}, {1431, {1, 1, 5, 3, 15, 55, 101, 67, 455, 625}},
    {1441, {1, 3, 5, 9, 1, 23, 29, 47, 345, 595}}, {1479, {1, 3, 7, 7, 5, 49, 29, 155, 323, 589}},
    {1509, {1, 3, 3, 7, 5, 41, 127, 61, 261, 717}}

};

struct SobolTable {
  uint32_t v[SOBOL_DIMS][SOBOL_BITS];
};

// V[d][j] = m_j 2^(31 - j), with m_j from the recurrence of the primitive polynomial of degree g (Bratley & Fox 1988;
// Joe & Kuo 2008): V[j] = V[j-g] ^ (V[j-g] >> g) ^ XOR over k = 1..g-1 of bit (g - k) of the polynomial times V[j-k].
constexpr SobolTable sobol_build() {
  SobolTable t{};
  for (int j = 0; j < SOBOL_BITS; ++j) t.v[0][j] = 1u << (31 - j);
  for (int d = 1; d < SOBOL_DIMS; ++d) {
    const uint32_t p = SOBOL_INIT[d].poly;
    int g = 0;
    while ((p >> (g + 1)) != 0) ++g;
    for (int j = 0; j < g; ++j) t.v[d][j] = SOBOL_INIT[d].m[j] << (31 - j);
    for (int j = g; j < SOBOL_BITS; ++j) {
      uint32_t v = t.v[d][j - g] ^ (t.v[d][j - g] >> g);
      for (int k = 1; k < g; ++k)
        if ((p >> (g - k)) & 1u) v ^= t.v[d][j - k];
      t.v[d][j] = v;
    }
  }
  return t;
}

constexpr SobolTable SOBOL_V = sobol_build();
#if defined(__CUDACC__)
__constant__ SobolTable sobol_v_dev = SOBOL_V;
#endif

SP_HD uint32_t sobol_v(int d, int j) {
#if defined(__CUDA_ARCH__)
  return sobol_v_dev.v[d][j];
#else
  return SOBOL_V.v[d][j];
#endif
}

// Coordinate d of point n as a 32-bit integer.  The loop runs over all 32 bits with a mask, so the lanes of a warp
// read the same direction number at every step (one broadcast from the constant cache).
SP_HD uint32_t sobol_coord(int d, uint32_t n) {
  const uint32_t g = n ^ (n >> 1);
  uint32_t x = 0;
  for (int j = 0; j < SOBOL_BITS; ++j) x ^= sobol_v(d, j) & (0u - ((g >> j) & 1u));
  return x;
}

SP_HD int sobol_slots(int K, int second_order) { return second_order ? 2 * K + 2 : K + 2; }

// Whether column j of design slot `slot` comes from B (the point's coordinate K + j) rather than A (coordinate j).
SP_HD int sobol_from_b(int K, int second_order, int slot, int j) {
  if (slot == 0) return 0;
  if (slot <= K) return slot - 1 == j;
  if (second_order && slot <= 2 * K) return slot - 1 - K != j;
  return 1;
}

// Value of free parameter j in design member m.
SP_HD double sobol_design_value(const SimplypSobol& sb, long long m, int j) {
  const int K = sb.n_free, P = sobol_slots(K, sb.second_order);
  const long long i = m / P;
  const int slot = (int)(m - i * P);
  const int d = sobol_from_b(K, sb.second_order, slot, j) ? K + j : j;
  const double u = (double)sobol_coord(d, (uint32_t)(sb.skip + i)) * (1.0 / 4294967296.0);
  const SimplypMcmcParam& p = sb.param[j];
  return mc_add(p.lo, mc_mul(mc_sub(p.hi, p.lo), u));
}

// The four words of bootstrap block q (draws 4q .. 4q + 3) of resample t.
SP_HD void sobol_boot_words(uint64_t seed, uint32_t t, uint32_t q, uint32_t (&r)[4]) {
  const uint32_t ctr[4] = {t, q, 0u, SOBOL_BLOCK};
  philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32), r);
}

// Position (0 .. n-1, in the row's used samples) that word w picks.
SP_HD uint32_t sobol_boot_pick(uint32_t w, uint32_t n) { return (uint32_t)(((uint64_t)w * n) >> 32); }

// Offset of pair (j, k), j < k, in the row-major upper triangle of a K x K matrix without its diagonal.
SP_HD int sobol_pair(int K, int j, int k) { return j * (2 * K - j - 1) / 2 + (k - j - 1); }

}  // namespace simplyp
