// simplyp_b200 — placement of a cost-ordered, latency-bound ensemble on the SMs: the arithmetic of the plan
// (which virtual blocks form which list, where a member of cost rank r sits).  Pure integer functions shared by the
// launcher, cost_scatter_kernel and plan_claim (simplyp_kernels.cu) and by the host-side test harness.
// At the end, launch_config(): the launch policy of the quad kernel (pilot, register variant, plan, epochs).
//
// B virtual blocks of 32 members, 2 resident blocks per SM on n_sm SMs.  With Q = max(0, B - 2 n_sm) virtual blocks
// too many for the machine, nY = n_sm - Q, nP = min(nY, B - nY - 3Q), xb = nY + nP:
//   first-list t < nY        : heavy virtual block t;                    its second-list: virtual block nY + t (t < nP)
//   first-list nY + x, x < Q : light blocks xb+Q+x then B-1-x (chained); its second-list: light block xb+x
// The launch has one block per list; a block claims its list by where it lands: the first block to arrive on an SM
// takes the next first-list, the second one the second-list that belongs to it (plan_claim).  cost_scatter_kernel
// With the 3-blocks-per-SM build (`resident` = 3) nothing is chained: the launch has 3 n_sm blocks, all resident at
// once; the Q SMs whose first block drew a ticket >= nY hold the three light blocks of a slot side by side (third-list
// 2 n_sm + nY + x = block B-1-x), the third block to arrive on any other SM has no list and leaves.  A slot that runs
// two light blocks one after the other ends late once the light blocks are more than half as heavy as the heaviest
// (measured after the day tolerance became rate-dependent: 10.4 ms against 8.2-8.7 ms for the other SMs).
// cost_scatter_kernel
// lays the members out so that virtual blocks [0, nY) are the heaviest in descending order, [nY, nY+nP) their
// partners in ASCENDING order (the heaviest block shares its SM with the lightest partner) and [xb, B) the 3Q
// lightest blocks in descending order (the two blocks that share a slot are taken from the lightest 2Q, a heavier
// one with a lighter one; the block beside them from the Q above).  So the hardware never queues a block (a queued
// block starts only when the first resident one ends, 7.6 ms into a 14 ms run at 10^4 members), and the two light
// blocks that must share a slot run beside a third light block that ends about when the first of them does.
#pragma once
#include <stdlib.h>

#include "simplyp_core.cuh"

namespace simplyp {

constexpr int FORC_TILE = 128;      // days per tile of the forcing ring (4 KB); epochs are whole tiles
constexpr int PLAN_MAX_SM = 1024;   // %smid is folded into this range

struct PlanShape {
  int n_sm, nY, nP, Q;
  int resident;                                            // blocks per SM the kernel build keeps resident: 2 or 3
  SP_HD int n_blocks() const { return nY + nP + 3 * Q; }
  SP_HD int n_lists() const { return resident == 3 ? n_blocks() : n_sm + nP + Q; }
  SP_HD int n_launch() const { return resident == 3 ? 3 * n_sm : n_lists(); }   // blocks of the launch
};

// Shape of the plan for B virtual blocks on n_sm SMs; false if the plan does not apply (B <= n_sm, or more than the
// lightest third of the resident set would have to be chained).
SP_HD bool plan_shape(long long B, int n_sm, PlanShape& p, int resident = 2) {
  if (n_sm <= 0 || B <= n_sm || B >= 3ll * n_sm) return false;
  const long long Q = B > 2ll * n_sm ? B - 2ll * n_sm : 0;
  const long long nY = n_sm - Q;
  if (nY <= 0) return false;
  long long nP = B - nY - 3 * Q;
  if (nP <= 0) return false;
  if (nP > nY) return false;                     // cannot happen for Q >= 0 (B <= 2 n_sm + Q), kept as a guard
  p.n_sm = n_sm; p.nY = (int)nY; p.nP = (int)nP; p.Q = (int)Q;
  p.resident = (resident == 3 && Q > 0) ? 3 : 2;
  return true;
}

// First virtual block of a list (-1: the list does not exist); lists [0, n_sm) are the first-lists, list n_sm + t is
// the second-list of first-list t, list 2 n_sm + t its third-list (resident = 3 only).
SP_HD int plan_list_head(const PlanShape& p, int list) {
  const int xb = p.nY + p.nP;
  if (list < 0) return -1;
  if (list < p.n_sm) return list < p.nY ? list : xb + p.Q + (list - p.nY);
  int t = list - p.n_sm;
  if (t < p.n_sm) {
    if (t < p.nY) return t < p.nP ? p.nY + t : -1;
    return xb + (t - p.nY);
  }
  t -= p.n_sm;
  if (p.resident != 3 || t < p.nY || t >= p.n_sm) return -1;
  return p.n_blocks() - 1 - (t - p.nY);
}
// virtual block that follows `vb` in its list, or -1
SP_HD int plan_list_next(const PlanShape& p, int vb) {
  if (p.resident == 3) return -1;
  const int x = vb - (p.nY + p.nP + p.Q);
  return (x >= 0 && x < p.Q) ? p.n_blocks() - 1 - x : -1;
}

// Member layout of a planned launch.  r = cost rank of a member (0 = heaviest); the result is its item index
// (virtual block = index / 32).
//  * the `solo` heaviest members each lead a warp of their own whose other seven quads hold light members (the
//    lightest of the partner region), so that the longest lock-step chain of the launch is one member's step count,
//    not the per-day maximum over eight similar heavy members;
//  * the blocks of the partner region [nY, nY + n_rev) are stored in reverse order (lightest first).
struct MemberLayout { int solo, nY, n_rev, fill_end; };

SP_HD MemberLayout member_layout(const PlanShape& p, int M, int solo) {
  MemberLayout L;
  if (8 * solo > 32 * p.nY || 7 * solo > 16 * p.nP || solo < 0) solo = 0;
  L.solo = solo;
  L.nY = p.nY;
  L.n_rev = p.nP - ((p.Q == 0 && M % 32 != 0) ? 1 : 0);      // a ragged last block stays last
  const long long pe = 32ll * (p.nY + p.nP);
  L.fill_end = (int)(pe < M ? pe : M);
  return L;
}

SP_HD int member_layout_index(int r, const MemberLayout& L) {
  const int K = L.solo, fill_begin = L.fill_end - 7 * K;
  if (r < K) return 8 * r;
  if (r >= fill_begin && r < L.fill_end) { const int t = r - fill_begin; return 8 * (t / 7) + 1 + t % 7; }
  if (r < fill_begin) r += 7 * K;
  const int blk = r >> 5;
  if (blk >= L.nY && blk < L.nY + L.n_rev) return ((L.nY + (L.n_rev - 1 - (blk - L.nY))) << 5) | (r & 31);
  return r;
}

// ------------------------------------------------------------------------------------------ launch policy
// How the launcher runs the quad kernel: whether a cost pilot runs, the register variant (MINB = resident blocks per
// SM) of every launch, the planned placement of an ensemble and the epochs of a network.  None of it changes a result.
struct LaunchInputs {
  int M, D;                   // members, days of the record
  bool network;               // false: an ensemble of one sub-catchment, whose items are the members
  int n_levels;               // network: topological levels
  long long grid_one_epoch;   // network: blocks of one pass over the items (the launcher's bound on the padded items)
  int pilot_days;             // SimplypOptions::pilot_days: 0 = 8 days, < 0 = no pilot
  bool workspace;             // the caller gave a workspace (the pilot hands its state over through it)
  int n_sm;
};
// SIMPLYP_<NAME> environment overrides, for A/B measurements (INTEGRATION.md §5).  0, -1 or false: the policy decides.
struct LaunchOverrides {
  int quad_minb = 0, pilot_minb = 0;      // QUAD_MINBLOCKS, PILOT_MINBLOCKS (2..4): an ensemble's main launch, pilot
  int net_minb = 0;                       // NET_MINBLOCKS (2, 3)
  bool no_plan = false;                   // SM_PLAN=0
  bool has_q_max = false; int q_max = 0;  // PLAN_QMAX: at most q_max SMs hold three blocks under the plan
  int solo = -1;                          // SOLO_WARPS (>= 0): warps led by one heavy member
  int epoch_days = -1;                    // EPOCH_DAYS, rounded down to whole tiles (<= 0 reads 0: one piece)
};
struct LaunchConfig {
  long long grid;             // blocks of the main launch (a network: of all its epochs)
  int minb;                   // variant of the main launch: simplyp_quad_kernel<MODE, minb, STIFF>
  int pilot_days, pilot_minb; // ensemble: days [0, pilot_days) are the cost pilot; 0: no pilot
  bool plan;                  // ensemble: planned placement (after the pilot)
  PlanShape shape;            // valid when plan
  int solo;                   // plan: led warps asked of member_layout()
  int epoch_days, n_epochs;   // network: 0 = one piece
};

inline LaunchOverrides read_launch_overrides() {
  LaunchOverrides o;
  int v = 0;
  const auto env = [&v](const char* name) { const char* e = getenv(name); v = e ? atoi(e) : 0; return e != nullptr; };
  if (env("SIMPLYP_QUAD_MINBLOCKS") && v >= 2 && v <= 4) o.quad_minb = v;
  if (env("SIMPLYP_PILOT_MINBLOCKS") && v >= 2 && v <= 4) o.pilot_minb = v;
  if (env("SIMPLYP_NET_MINBLOCKS") && (v == 2 || v == 3)) o.net_minb = v;
  o.no_plan = env("SIMPLYP_SM_PLAN") && v == 0;
  if ((o.has_q_max = env("SIMPLYP_PLAN_QMAX"))) o.q_max = v;
  if (env("SIMPLYP_SOLO_WARPS") && v >= 0) o.solo = v;
  if (env("SIMPLYP_EPOCH_DAYS")) o.epoch_days = v > 0 ? v / FORC_TILE * FORC_TILE : 0;
  return o;
}

inline LaunchConfig launch_config(const LaunchInputs& in, const LaunchOverrides& o) {
  LaunchConfig c{};
  const long long n_sm = in.n_sm;
  if (!in.network) {
    c.grid = (in.M + 31ll) / 32;                         // 32 members per block
    // Every block resident at 2 per SM (184 registers).  Beyond that the 168-register build (3 blocks per SM, no
    // spills) up to about 4x10^4 members; the 128-register build (4 blocks per SM, 136 B of spills in the step loop)
    // only where the machine is several waves deep.  Round 2, B200, 3 vs 4 blocks: 2x10^4 members 19.6 vs 20.9 ms,
    // 4x10^4 35.1 vs 35.3, 1.6x10^5 131.7-132.0 vs 130.3-131.1.
    c.minb = o.quad_minb ? o.quad_minb : c.grid <= 2 * n_sm ? 2 : c.grid <= 9 * n_sm ? 3 : 4;
    const int days = in.pilot_days > 0 ? in.pilot_days : 8;
    if (in.pilot_days < 0 || !in.workspace || in.M < 512 || in.D < 8 * days) return c;
    c.pilot_days = days;
    // register variant of the pilot pass (the variants give the same bits): when the 2-blocks-per-SM build would leave
    // a few blocks queued behind the resident ones, the 3-blocks build runs them all at once
    c.pilot_minb = o.pilot_minb ? o.pilot_minb : (c.minb == 2 && c.grid > 2 * n_sm) ? 3 : c.minb;
    // latency-bound regime (every block resident at once: 2 per SM, or 3 on some SMs with the 168-register build):
    // planned placement.  B200, round 2, planned / unplanned 3-blocks launch: 10^4 members 9.4 / 11.6 ms,
    // 1.2x10^4 11.0 / 12.0, 1.4x10^4 12.0 / 12.5 (the chained 2-blocks plan of round 1: 10.8 / 12.5 / 13.4).
    const long long q_max = o.has_q_max ? o.q_max : n_sm - 1;
    c.plan = (c.minb == 2 || (c.minb == 3 && c.grid <= 2 * n_sm + q_max)) && n_sm <= PLAN_MAX_SM && in.M >= 2048 &&
             !o.no_plan && plan_shape(c.grid, in.n_sm, c.shape, c.minb);
    if (c.plan) {
      c.solo = o.solo >= 0 ? o.solo : in.M / 100 / 4 * 4;   // about one warp in five of the heavy blocks (10^4 members:
                                                             // 0 / 24 / 96 / 240 led warps 9.55 / 9.42 / 9.35 / 9.51 ms)
      c.grid = c.shape.n_launch();   // fills the resident slots: one block per list at 2 per SM, 3 n_sm blocks at 3
    }
    return c;
  }
  // Epoch sweep (KArgs::epoch_days): a whole number of forcing tiles per epoch.  Without it the launch is the bulk of
  // the headwaters followed by the chains of the main-stem reaches at low occupancy.  An epoch should be long against
  // the depth of the network (the wavefront needs one day-time per level to reach the outlet): four days per level,
  // at least 256.  B200, round 2, one piece / 256 / 512 / 1024 / 2048 days per epoch: config 3 (32 levels) at 64
  // members 767 / 555 / 564 / 567 / 583 ms, at 256 members 2185 / 1922 / 1920 / 1932 / 1929; config 5 (487 levels) at
  // 8 members 2565 / 2788 / 2550 / 2411 / 2348 ms, at 1 member 1339 / 1297 / 1244 / 1253 / 1279.
  int epoch_days = (4 * in.n_levels + FORC_TILE - 1) / FORC_TILE * FORC_TILE;
  if (epoch_days < 2 * FORC_TILE) epoch_days = 2 * FORC_TILE;
  // a launch of at most one block per SM has no bulk phase to overlap with, and its chain warps have their SMs to
  // themselves: swept in epochs they would only get neighbours (config 3 at 1 / 8 members, 15 / 72 blocks: 549 / 548
  // ms in one piece, 590 / 573 in epochs; config 5 at 1 member, 227 blocks, still gains: 1394 -> 1307 ms)
  if (in.grid_one_epoch <= n_sm) epoch_days = 0;
  if (o.epoch_days >= 0) epoch_days = o.epoch_days;
  c.grid = in.grid_one_epoch;
  if (epoch_days > 0 && in.D > epoch_days && c.grid * ((in.D + epoch_days - 1) / epoch_days) < (1ll << 30)) {
    c.epoch_days = epoch_days;
    c.n_epochs = (in.D + epoch_days - 1) / epoch_days;
    c.grid *= c.n_epochs;
  }
  // Networks get the build with the Rosenbrock path for stiff (main-stem) reaches.  Its 2-blocks-per-SM variant (226
  // registers) serves launches that the chains of the main stem bound; when the items of one epoch fill the machine
  // several times over, the 3-blocks variant (168 registers, 40 B of spills) is faster.  B200, round 2, 2 / 3 blocks:
  // config 3 at 64 members (512 blocks per epoch) 557 / 666 ms, at 256 members (2048) 1921 / 1739; config 5 at 8
  // members (1024) 2346 / 2166, at 1 member (128) 1266 / 1583.
  c.minb = o.net_minb ? o.net_minb : in.grid_one_epoch >= 6 * n_sm ? 3 : 2;
  return c;
}

}  // namespace simplyp
