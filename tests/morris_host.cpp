// TEST HARNESS ONLY — compiles simplyp_morris.cuh (the trajectories, design values, trajectory distances, greedy
// selection and bootstrap picks of the Morris screening) for the host, so that the CPU-only test tier can check it
// against NumPy without a GPU.  Nothing in simplyp_b200/ loads this library; the product has no CPU execution path.
#include <cmath>
#include <cstdint>
#include <vector>

#include "../simplyp_b200/csrc/simplyp_morris.cuh"

using namespace simplyp;

// Levels of candidates c0 .. c0 + n - 1: out[n][K + 1][K].
extern "C" void morris_host_levels(uint64_t seed, int64_t c0, int64_t n, int K, int p, int32_t* out) {
  std::vector<uint8_t> t(4 * K);
  for (int64_t c = 0; c < n; ++c) {
    morris_traj_pack(seed, (uint32_t)(c0 + c), K, p, t.data());
    for (int s = 0; s <= K; ++s)
      for (int z = 0; z < K; ++z) out[(c * (K + 1) + s) * K + z] = morris_level(t.data(), K, p / 2, s, z);
  }
}

// Values of the K free parameters of design members member_offset .. member_offset + n - 1: out[n][K]
// (selected may be NULL: trajectory i is candidate i).
extern "C" void morris_host_design(const SimplypMorris* mo, const int32_t* selected, int64_t member_offset, int64_t n,
                                   double* out) {
  const int K = mo->n_free, p = mo->num_levels;
  std::vector<uint8_t> t(4 * K);
  for (int64_t q = 0; q < n; ++q) {
    const int64_t m = member_offset + q, i = m / (K + 1);
    const int s = (int)(m - i * (K + 1));
    morris_traj_pack(mo->seed, (uint32_t)(selected ? selected[i] : i), K, p, t.data());
    for (int j = 0; j < K; ++j) out[q * K + j] = morris_value(mo->param[j], morris_level(t.data(), K, p / 2, s, j), p);
  }
}

// The greedy selection of n_trajectories among n_candidates: selected[r].
extern "C" void morris_host_select(const SimplypMorris* mo, int32_t* selected) {
  const int K = mo->n_free, p = mo->num_levels, nc = mo->n_candidates, r = mo->n_trajectories;
  std::vector<uint8_t> t((size_t)nc * 4 * K);
  for (int c = 0; c < nc; ++c) morris_traj_pack(mo->seed, (uint32_t)c, K, p, t.data() + (size_t)c * 4 * K);
  auto dist = [&](int a, int b) {
    return a < b ? morris_distance(t.data() + (size_t)a * 4 * K, t.data() + (size_t)b * 4 * K, K, p / 2)
                 : morris_distance(t.data() + (size_t)b * 4 * K, t.data() + (size_t)a * 4 * K, K, p / 2);
  };
  double best = -1.0;
  for (int m = 0; m < nc; ++m)
    for (int l = m + 1; l < nc; ++l) {
      const double d = dist(m, l);
      if (d > best) best = d, selected[0] = m, selected[1] = l;
    }
  std::vector<double> score(nc, 0.0);
  std::vector<char> in(nc, 0);
  in[selected[0]] = in[selected[1]] = 1;
  for (int k = 0; k + 1 < r; ++k) {
    const int s = selected[k];
    for (int c = 0; c < nc; ++c)
      if (!in[c]) {
        const double d = dist(c, s);
        score[c] = score[c] + d * d;
      }
    if (k == 0) continue;
    int arg = -1;
    for (int c = 0; c < nc; ++c)
      if (!in[c] && (arg < 0 || score[c] > score[arg])) arg = c;
    selected[k + 1] = arg;
    in[arg] = 1;
  }
}

// Positions (in n used trajectories) of the draws 0 .. count - 1 of bootstrap resample b: out[count].
extern "C" void morris_host_picks(uint64_t seed, uint32_t b, uint32_t n, int64_t count, uint32_t* out) {
  for (int64_t k = 0; k < count; k += 4) {
    uint32_t w[4];
    morris_words(seed, b, (uint32_t)(k / 4), 1u, w);
    for (int q = 0; q < 4 && k + q < count; ++q) out[k + q] = morris_pick(w[q], n);
  }
}
