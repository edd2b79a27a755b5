// simplyp_kernels.cu — sm_100a kernels and the C-ABI of simplyp_b200 (see include/simplyp_b200.h).
//
// Kernels
//   simplyp_quad_kernel<MODE,MINB,STIFF>  K1 (+K1a TMA forcing ring, K1b reach routing, K2 output writer or K3 fused
//                                   statistics): a quad of 4 lanes per (ensemble member, sub-catchment), 8 quads per
//                                   warp in day lock-step; replaces the reference's SC x day loop body,
//                                   model.py:365-724 (program: simplyp_quad.cuh, day-boundary algebra: simplyp_core.cuh)
//   stiff_group_kernel              per-reach stiffness estimate that orders the reaches of a level (device side, so
//                                   that the *_device entry points never synchronise)
//   cost_scan_kernel, cost_scatter_kernel  counting sort of the pilot costs (member order of an ensemble)
//   obs_const_kernel, obs_rank_kernel, spearman_kernel  observation constants / Spearman's r of
//                                   goodness_of_fit_stats (visualise_results.py:441-449)
//   waterbody_kernel                sum_to_waterbody (model.py:851-900)
//   thornthwaite_kernel             daily_PET (inputs.py:232-312)
//   fp64_peak_kernel, fp64_latency_kernel  DFMA throughput / latency probes for the roofline denominator
//   mcmc_propose_kernel, mcmc_accept_kernel, mcmc_advance_kernel, mcmc_init_kernel  ensemble sampler (stretch move,
//                                   arithmetic in simplyp_mcmc.cuh) over the fused log-likelihood
//   predictive_draws_kernel         posterior predictive draws of the simulated series (simplyp_bands.cuh)
//   nanquantile_kernel, nq_prepare_kernel, nq_hist_kernel, nq_pick_kernel  np.nanquantile of the rows of a matrix
//
// There is deliberately no host implementation of the integration in this library.
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include "simplyp_quad.cuh"
#include "simplyp_plan.cuh"
#include "simplyp_mcmc.cuh"
#include "simplyp_bands.cuh"

using namespace simplyp;

namespace {

// ------------------------------------------------------------------------------------------ errors
thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, const char* detail = "") {
  snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}

#define SP_CUDA(call)                                                            \
  do {                                                                           \
    cudaError_t e__ = (call);                                                    \
    if (e__ != cudaSuccess) {                                                    \
      snprintf(g_err, sizeof(g_err), "%s failed: %s", #call, cudaGetErrorString(e__)); \
      return (e__ == cudaErrorMemoryAllocation) ? SIMPLYP_ENOMEM : SIMPLYP_ECUDA; \
    }                                                                            \
  } while (0)

__device__ int g_zero_offsets[2] = {0, 0};   // CSR offsets of a network without edges

// ------------------------------------------------------------------------------------------ kernel args
struct KArgs {
  int M, S, D, Msc, V;
  ThreadOptions topt;
  int sc_qr0;
  const double* forcing;        // [D][4]
  const double* member_params;  // [M][NP_MEMBER]
  const double* sc_params;      // [Msc][S][NP_SC]
  const int* parent_offsets;    // [S+1]   (device copy)
  const int* parent_ids;        // [E]
  const int* work_sc;           // sub-catchments handled by this launch
  int n_work;
  double* out;                  // run: [M][S][D][25]
  long long* diag;              // [M][S][4] or null
  const double* obs;            // cal: [V][D]
  const int* obs_desc;          // cal: [V][2]
  const double* obs_const;      // cal: [V][8]
  const double* obs_log;        // cal: [V][D] natural log of the observations (NaN where there is none), or null
  double* stats;                // cal: [M][V][8]
  double* flux;                 // cal, S>1: [M][S][D][4]
  int* progress;                // S>1: [M][S] days completed (release/acquire flags of the routing wavefront)
  int* ticket;                  // S>1: block ticket counter (virtual block order = dispatch order)
  // quad kernel, S>1: items (reach, member) are laid out level by level, each level padded to a multiple of
  // 8 items so that the 8 quads of a lock-step warp never depend on each other
  const long long* level_item_off;  // [n_levels+1] padded cumulative item counts
  const int* level_order_off;       // [n_levels+1] offsets into work_sc
  int n_levels;                     // the padded item total is level_item_off[n_levels] (device side)
  // cost ordering of an ensemble (quad kernel, one sub-catchment): a short pilot run counts the step attempts
  // of every member; members are then dealt to the lock-step warps heaviest first
  double* sim_obs;              // cal + rank statistics: [M][V][D] simulated value on observed days, or null
  const int* perm;              // [M] member handled by item idx, or null
  unsigned* cost;               // pilot: [M] step attempts
  unsigned* hist;               // pilot: [COST_BUCKETS] histogram of the costs
  // The pilot is the FIRST PART of the run: the same kernel integrates days [0, pilot days) in member order, stores
  // every member's midnight state (carry) and its step attempts (cost); the main launch continues at day_begin.
  QuadCarry* carry;             // [M] or null
  double* carry_stats;          // cal: [M][STAT_SLOTS * RS_COUNT] shared-memory fit-statistic sums at the hand-over, or null
  int day_begin;                // first day this launch integrates (main launch after a pilot), else 0
  int day_end;                  // one past the last day this launch integrates (D, or the pilot's days); D stays the
                                // length of the record, i.e. the stride of forcing / obs / out
  int pilot_pass;               // 1: this launch is the pilot (writes cost / hist / carry, no diagnostics, no finalise)
  // Networks: the record is cut into epochs of epoch_days days and the launch sweeps (epoch, block of items) units in
  // epoch-major ticket order, the midnight state of every item crossing an epoch boundary through `carry` (indexed
  // [m][s]): the chains of the main-stem reaches of epoch e then run beside the headwaters of epoch e+1 instead of
  // alone at the end of the launch.  0 = one epoch.
  int epoch_days, n_epochs;
  int* epoch_done;              // [M][S] epochs an item has completed (release/acquire, like `progress`)
  // *_host entry points stream the rows of a finished epoch to the caller's buffer while later epochs integrate: the
  // last item to finish epoch e raises epoch_flags_host[e] (mapped pinned memory), which the host thread polls
  unsigned* epoch_count;        // [n_epochs] items that have finished the epoch, or null
  int* epoch_flags_host;        // [n_epochs] device pointer of the mapped flags, or null
  // calibration fused with the all-gather of the statistics (simplyp_calibrate_gather_device): every rank's gather
  // buffer as mapped into this process; finalise() stores a member's statistics into all of them
  double* peer_stats[SIMPLYP_MAX_RANKS];
  int n_peers, my_rank;         // n_peers = 0: no gather
  long long member_offset;      // this rank's first member in the buffers
  int* plan;                    // placement of a cost-ordered ensemble on the SMs (PLAN_* below), or null
  PlanShape shape;              // valid when plan != nullptr
};
constexpr int COST_BUCKETS = 4096;

// Placement plan (simplyp_plan.cuh): device-side bookkeeping of the claims, an int array in the workspace.
constexpr int PLAN_FIRST_NEXT = 0;
constexpr int PLAN_SKIPS = 1;                      // blocks that left without a list (launches with more blocks than lists)
constexpr int PLAN_SM_ARR = 16;                    // [PLAN_MAX_SM] blocks that have arrived on the SM
constexpr int PLAN_SM_LIST = PLAN_SM_ARR + PLAN_MAX_SM;         // [PLAN_MAX_SM] 1 + first-list of the SM, -1: none
constexpr int PLAN_CLAIMED = PLAN_SM_LIST + PLAN_MAX_SM;        // [3 * PLAN_MAX_SM] list taken?
constexpr int PLAN_INTS = PLAN_CLAIMED + 3 * PLAN_MAX_SM;       // zeroed before every launch

// raw sums kept in stats[][][] while a calibration kernel runs (finalised in place at the end).  S1, S2 and SOS are
// taken about RS_SHIFT, the simulated value of the series' first observed day (fixed there, carried with the sums).
enum { RS_N = 0, RS_SSE, RS_SSE_LOG, RS_LL, RS_S1, RS_S2, RS_SOS, RS_SABS, RS_SHIFT, RS_COUNT };
static_assert((int)RS_COUNT <= (int)SIMPLYP_NSTAT, "the raw sums of a series beyond STAT_SLOTS live in its stats row");
// obs_const[V][8]
enum { OC_N = 0, OC_MEAN, OC_SS, OC_MEAN_LOG, OC_SS_LOG, OC_SUM, OC_STD, OC_SS_RANK };

// ------------------------------------------------------------------------------------------ K1a forcing ring
// The daily forcing (32 B/day, shared by every member and sub-catchment) is staged per block in a ring of
// FORC_SLOTS shared-memory tiles of FORC_TILE days each, filled by 1-D TMA bulk copies
// (cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes) that signal one mbarrier per slot.
// There is no producer warp: threads walk through the days at their own pace, and the LAST thread of the
// block to leave tile k re-arms the slot and issues the copy of tile k+FORC_SLOTS into it.  A thread that
// runs ahead of the ring polls (mbarrier.test_wait) once per loop iteration instead of blocking, so the
// slowest thread — which is always inside a resident tile — is never held up.  FORC_TILE: simplyp_plan.cuh.
constexpr int FORC_SLOTS = 4;     // ring depth (16 KB per block)

struct ForcingRing {
  double tiles[FORC_SLOTS][FORC_TILE * SIMPLYP_NF];
  unsigned long long full[FORC_SLOTS];   // mbarriers
  unsigned left[FORC_SLOTS];             // warps that have left the tile currently held by the slot
  unsigned n_consumers;
  int first_tile;                        // tile of the first day this launch integrates (slot = (tile - first) % SLOTS)
  int end_day;                           // one past the last day this launch reads: no tile at or beyond it is fetched
};

__device__ __forceinline__ int ld_acquire_s32(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned smem_u32(const void* p) {
  return static_cast<unsigned>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_inval(unsigned long long* bar) {
  asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_test_parity(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// arm the barrier with the byte count and start the bulk copy global -> shared
__device__ __forceinline__ void tma_load_tile(ForcingRing* ring, int slot, const double* forcing, int tile, int n_days) {
  const int d0 = tile * FORC_TILE;
  const int nd = (n_days - d0) < FORC_TILE ? (n_days - d0) : FORC_TILE;
  const unsigned bytes = (unsigned)nd * SIMPLYP_NF * sizeof(double);
  const unsigned bar = smem_u32(&ring->full[slot]);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // earlier generic reads of the slot are done
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(&ring->tiles[slot][0])), "l"(forcing + (size_t)d0 * SIMPLYP_NF), "r"(bytes), "r"(bar)
               : "memory");
}

// ------------------------------------------------------------------------------------------ IO policies
// ROUTED = the network build of the kernel (reach routing: progress flags, parents' fluxes).  It is a compile-time
// property on purpose: an ensemble of one sub-catchment must not even contain the routing loops — besides their cost,
// control flow whose convergence ptxas cannot prove (loops over a thread's own parent list that are left from the
// middle, the per-thread level search) made it guard EVERY quad shuffle of the step loop with a divergence check and
// copy each shuffled register pair (673 instead of ~600 instructions per step attempt, profiles/r02_step_loop.sass).
template <bool ROUTED>
struct IOBase {
  const KArgs& a;
  int m, s;
  const double* scp_member;  // this member's [S][NP_SC] block
  ForcingRing* ring;
  int my_tile;               // tile this thread currently reads from (-1 before the first day)
  int wait_status;           // status bits raised by wait()
  __device__ IOBase(const KArgs& a_, int m_, int s_, ForcingRing* ring_)
      : a(a_), m(m_), s(s_), scp_member(a_.sc_params + (size_t)(a_.Msc > 1 ? m_ : 0) * a_.S * SIMPLYP_NP_SC),
        ring(ring_), my_tile(-1), wait_status(0) {}

  // The warp enters the forcing tile of `day` (all lanes call it with the same `day`; the ring's consumers are the
  // warps of the block and lane 0 does the bookkeeping): on a tile change it first leaves its old tile — the last
  // warp out re-arms the slot and starts the copy of tile k+FORC_SLOTS into it — and then waits for the new tile's
  // mbarrier.  Every branch and loop condition here is a warp vote, i.e. provably warp-uniform: with thread-varying
  // conditions around the lane-0 region ptxas could not prove the warp converged afterwards and guarded every
  // shuffle of the step loop with a divergence check plus register copies (+12 % instructions per step attempt).
  __device__ __forceinline__ bool enter_tile(int day, long long t0, long long limit) {
    const int q = day / FORC_TILE;
    if (__any_sync(0xffffffffu, q != my_tile)) {
      if (__any_sync(0xffffffffu, my_tile >= 0 && my_tile == q - 1)) {
        __syncwarp();                                         // every lane is done reading the old tile
        if ((threadIdx.x & 31) == 0) {
          const int slot = (my_tile - ring->first_tile) % FORC_SLOTS;
          const unsigned before = atomicAdd(&ring->left[slot], 1u);
          if (before + 1 == ring->n_consumers) {
            ring->left[slot] = 0;
            const int next = my_tile + FORC_SLOTS;
            if (next * FORC_TILE < ring->end_day) tma_load_tile(ring, slot, a.forcing, next, a.D);
          }
        }
        __syncwarp();
      }
      const int rel = q - ring->first_tile;
      bool ok = true;
      while (ok && !__all_sync(0xffffffffu, mbar_test_parity(&ring->full[rel % FORC_SLOTS], (unsigned)(rel / FORC_SLOTS) & 1u)))
        ok = __all_sync(0xffffffffu, (clock64() - t0) < limit);
      my_tile = q;
      return ok;
    }
    return true;
  }
  // upstream reaches of this item have published `day`?  The loop over the item's own parent list runs a
  // WARP-UNIFORM number of times (the longest list in the warp, lanes past their own list idle): a loop whose trip
  // count varies between the lanes is another shape that costs ptxas its convergence proof (see IOBase).
  __device__ __forceinline__ bool upstream_ready(int day) const {
    const int e0 = a.parent_offsets[s], n = a.parent_offsets[s + 1] - e0;
    const int n_max = __reduce_max_sync(0xffffffffu, n);
    int oldest = 0x7fffffff;
    for (int k = 0; k < n_max; ++k) {
      if (k < n) {
        const int* flag = a.progress + (size_t)m * a.S + a.parent_ids[e0 + k];
        int done;
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(done) : "l"(flag) : "memory");
        oldest = done < oldest ? done : oldest;
      }
    }
    return oldest > day;
  }
  // quad program: block (the whole warp) until forcing and upstream inputs of `day` exist
  // A watchdog (2^37 cycles, about 70 s of SM clock) turns a wait that can never end (a bug, or a launch that
  // violates the dispatch-order argument) into status bit 2 instead of a hung device.  A legitimate wait is short:
  // the parents of a reach were dispatched earlier and are resident or finished, so a warp of topological level L
  // waits at most about L day-times at the start of the run (a chain of 10^5 reaches: ~3 s) and a day-time after.
  __device__ __forceinline__ void wait(int day) {
    const long long limit = 1ll << 37;
    const long long t0 = clock64();
    bool ok = enter_tile(day, t0, limit);
    if (ROUTED && a.progress != nullptr) {
      unsigned ns = 32;
      while (ok && !__all_sync(0xffffffffu, upstream_ready(day))) {
        __nanosleep(ns);
        if (ns < 1024) ns *= 2;
        ok = __all_sync(0xffffffffu, (clock64() - t0) < limit);
      }
    }
    if (!ok) wait_status |= 4;
  }

  // release store that pairs with the acquire load in upstream_ready()
  __device__ __forceinline__ void publish(int day) const {
    if (!ROUTED || a.progress == nullptr) return;
    int* flag = a.progress + (size_t)m * a.S + s;
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(flag), "r"(day + 1) : "memory");
  }

  __device__ __forceinline__ void forcing(int day, double& P, double& E, double& doy, double& T_air) const {
    const double* f = &ring->tiles[(day / FORC_TILE - ring->first_tile) % FORC_SLOTS][(day % FORC_TILE) * SIMPLYP_NF];
    P = f[0];
    E = f[1];
    doy = f[2];
    T_air = f[3];
  }
};

// Full-output mode: parents' fluxes are read back from their output rows (columns Qr, Msus_kg/day,
// TDP_kg/day, PP_kg/day — exactly what the reference reads from df_R_dict, model.py:524-528).
template <bool ROUTED>
struct RunIO : IOBase<ROUTED> {
  using B = IOBase<ROUTED>;
  using B::a; using B::m; using B::s; using B::scp_member;
  __device__ RunIO(const KArgs& a_, int m_, int s_, ForcingRing* ring_) : B(a_, m_, s_, ring_) {}
  __device__ __forceinline__ void upstream(int day, double (&us)[4]) const {
    us[0] = us[1] = us[2] = us[3] = 0.0;
    if (!ROUTED) return;
    const int e0 = a.parent_offsets[s], n = a.parent_offsets[s + 1] - e0;
    const int n_max = __reduce_max_sync(0xffffffffu, n);       // warp-uniform trip count, see upstream_ready()
    const double A_this = scp_member[(size_t)s * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
    const double rA_this = sp_rcp(A_this);             // (A_up / A_this by sp_div: no division subroutine in the day loop)
    for (int k = 0; k < n_max; ++k) {
      if (k < n) {
        const int p = a.parent_ids[e0 + k];
        const double* row = a.out + (((size_t)m * a.S + p) * a.D + day) * SIMPLYP_NOUT;
        const double A_up = scp_member[(size_t)p * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
        us[0] += __ldcg(row + SIMPLYP_O_QR) * sp_div(A_up, A_this, rA_this);   // :525
        us[1] += __ldcg(row + SIMPLYP_O_MSUS_FLUX);
        us[2] += __ldcg(row + SIMPLYP_O_TDP_FLUX);
        us[3] += __ldcg(row + SIMPLYP_O_PP_FLUX);
      }
    }
  }
  // K2: the 200-byte output row out[m][s][day][0:25] (the reference's 12 + 13 raw columns, model.py:737-745).  Every
  // lane of the quad holds the whole row (the day-boundary algebra is redundant across the quad), so the four lanes
  // store it together: lane l writes columns l, l+4, l+8, ... — each store instruction of the warp moves eight
  // contiguous 32-byte pieces (one per quad) instead of eight single doubles, 7 store instructions per day instead
  // of 25 by the leader alone.  The column a lane stores is chosen with selects, not by indexing a register array.
  static constexpr bool kAllLanesEmit = true;
  template <class Q>
  __device__ __forceinline__ void emit(const Q& q, int day, const double (&y)[NL], double Vr, const double (&acc)[NA],
                                       const double (&non)[13], const Cold&) const {
    double* row = a.out + (((size_t)m * a.S + s) * a.D + day) * SIMPLYP_NOUT + q.ql;
    const double r[28] = {y[iVsA], y[iVsS], y[iVg], Vr, y[iQr], acc[0], y[iMsus], acc[1], y[iTDPr], acc[2], y[iPPr], acc[3],
                          non[0], non[1], non[2], non[3], non[4], non[5], non[6], non[7], non[8], non[9], non[10], non[11],
                          non[12], 0.0, 0.0, 0.0};
    static_assert(SIMPLYP_O_QQ == 12 && SIMPLYP_NOUT == 25 && SIMPLYP_O_VR == 3 && SIMPLYP_O_PP_FLUX == 11, "row layout");
#pragma unroll
    for (int i = 0; i < 6; ++i) row[4 * i] = q.pick(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
    if (q.ql == 0) row[24] = r[24];
  }
};

// Calibration mode: nothing is written per day except (for S>1) the 4 fluxes the downstream reach
// needs; observed days update the running sums of the fit statistics.
// Running sums of the fit statistics of one (member, sub-catchment) item.  The quad kernel keeps them in SHARED
// memory (STAT_SLOTS series per item: a reach has at most the six kinds Q, SS, TDP, PP, TP, SRP): the per-day
// read-modify-write of eight sums per series in global memory was the largest stall of the day-boundary code.
// Series beyond STAT_SLOTS on one reach, and the one-thread-per-item kernel, accumulate in stats[][][] directly.
constexpr int STAT_SLOTS = 6;
constexpr int STAT_STRIDE = STAT_SLOTS * RS_COUNT + 1;   // doubles per item; odd: the 8 quad leaders of a warp hit distinct banks
static_assert(STAT_SLOTS * RS_COUNT % 2 == 0, "the accumulators are zeroed / restored in pairs");
// The calibration launches of simplyp_quad_kernel (32 quads a block) do not opt in to more than the default 48 KB of
// shared memory a block: quad state, forcing ring and these accumulators (dynamic) plus the exp2 table (static).
static_assert(32 * sizeof(QuadMem) + sizeof(ForcingRing) + 32 * STAT_STRIDE * sizeof(double) +
                  EXP_TAB * sizeof(double) + 2 * sizeof(int) <= 48 * 1024,
              "calibration shared memory above 48 KB a block: opt in with cudaFuncAttributeMaxDynamicSharedMemorySize");

template <bool ROUTED>
struct CalIO : IOBase<ROUTED> {
  using B = IOBase<ROUTED>;
  using B::a; using B::m; using B::s; using B::scp_member;
  double f_TDP;
  double* sacc;     // shared-memory accumulators of this item [STAT_SLOTS][RS_COUNT], or null
  __device__ CalIO(const KArgs& a_, int m_, int s_, ForcingRing* ring_, double f_TDP_, double* sacc_ = nullptr)
      : B(a_, m_, s_, ring_), f_TDP(f_TDP_), sacc(sacc_) {}

  __device__ __forceinline__ void upstream(int day, double (&us)[4]) const {
    us[0] = us[1] = us[2] = us[3] = 0.0;
    if (!ROUTED) return;
    const int e0 = a.parent_offsets[s], n = a.parent_offsets[s + 1] - e0;
    const int n_max = __reduce_max_sync(0xffffffffu, n);       // warp-uniform trip count, see upstream_ready()
    const double A_this = scp_member[(size_t)s * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
    const double rA_this = sp_rcp(A_this);             // (A_up / A_this by sp_div: no division subroutine in the day loop)
    for (int k = 0; k < n_max; ++k) {
      if (k < n) {
        const int p = a.parent_ids[e0 + k];
        const double* row = a.flux + (((size_t)m * a.S + p) * a.D + day) * 4;
        const double A_up = scp_member[(size_t)p * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
        us[0] += __ldcg(row + 0) * sp_div(A_up, A_this, rA_this);
        us[1] += __ldcg(row + 1);
        us[2] += __ldcg(row + 2);
        us[3] += __ldcg(row + 3);
      }
    }
  }
  static constexpr bool kAllLanesEmit = false;
  template <class Q>
  __device__ __forceinline__ void emit(const Q&, int day, const double (&)[NL], double, const double (&acc)[NA],
                                       const double (&)[13], const Cold& c) const {
    if (a.flux != nullptr) {
      double* row = a.flux + (((size_t)m * a.S + s) * a.D + day) * 4;
      row[0] = acc[0]; row[1] = acc[1]; row[2] = acc[2]; row[3] = acc[3];
    }
    // simulated counterparts of the observed series (sim_series_value, simplyp_bands.cuh) in the reference's own order
    // of operations (model.py:784-793, :840-845): Q_cumecs = Qr*A*1000/86400, concentrations (flux/Qr)/A_catch.
    // The quotients are formed by sp_div (reciprocal, product, one fma of the exact remainder: the IEEE quotient in
    // all but rare last-bit cases) because
    // Spearman's r is sensitive to the last bit wherever simulated values tie (recession days at the groundwater floor:
    // 2e-6 on 13,700 pairs between two orders of evaluation).  A true IEEE division would bring its slow-path
    // subroutine into the kernel: its mere presence, never executed, cost 2-3 % of the run time (A/B on one box).
    const double A = c.A_catch;
    const double rQ = sp_rcp(acc[0]), rA = sp_rcp(A);
    int slot = 0;
    for (int v = 0; v < a.V; ++v) {
      if (__ldg(a.obs_desc + 2 * v) != s) continue;
      const int k = slot++;
      const double o = __ldg(a.obs + (size_t)v * a.D + day);
      if (o != o) continue;  // no observation that day
      const int kind = __ldg(a.obs_desc + 2 * v + 1);
      const double sim = sim_series_value(kind, acc[0], acc[1], acc[2], acc[3], A, rQ, rA, f_TDP);   // (predictive_draws_kernel too)
      if (a.sim_obs != nullptr) a.sim_obs[((size_t)m * a.V + v) * a.D + day] = sim;
      const double* oc = a.obs_const + 8 * v;
      const double mo = __ldg(oc + OC_MEAN);
      const double em = __ldg(a.member_params + (size_t)m * SIMPLYP_NP_MEMBER + SIMPLYP_P_ERR_M0 + kind);
      const double d = o - sim;
      const double sg = em * sim;
      // natural logs: of the observation precomputed once per run; of the simulated value by the branch-free
      // sp_log, which needs a positive argument (anything else gives NaN, i.e. -inf log-likelihood, as np.log does)
      const double lo = a.obs_log ? __ldg(a.obs_log + (size_t)v * a.D + day) : log(o);
      const double ls = (sim > 0.0) ? sp_log(sim) : NAN;
      const double lsg = (sg > 0.0) ? sp_log(sg) : NAN;
      const double dl = lo - ls;
      const double rsg = sp_rcp(sg);
      double* rs = (sacc != nullptr && k < STAT_SLOTS) ? sacc + RS_COUNT * k
                                                       : a.stats + ((size_t)m * a.V + v) * SIMPLYP_NSTAT;
      // the simulated-side sums about a shift near the simulated series, not about mean(obs): S2 - S1^2/n then keeps
      // its digits when the two means are far apart (observations in other units, a flat offset member)
      const double n0 = rs[RS_N];
      const double shift = (n0 == 0.0) ? sim : rs[RS_SHIFT];
      rs[RS_SHIFT] = shift;
      const double ds = sim - shift;
      rs[RS_N] = n0 + 1.0;
      rs[RS_SSE] += d * d;
      rs[RS_SSE_LOG] += dl * dl;
      rs[RS_LL] += -0.91893853320467274178 - lsg - 0.5 * (d * rsg) * (d * rsg);   // MCMC.ipynb:233-236
      rs[RS_S1] += ds;
      rs[RS_S2] += ds * ds;
      rs[RS_SOS] += (o - mo) * ds;
      rs[RS_SABS] += fabs(d);
    }
  }
  // turn the raw sums of this item's series into the statistics of visualise_results.py:441-449
  __device__ void finalise() const {
    int slot = 0;
    for (int v = 0; v < a.V; ++v) {
      if (a.obs_desc[2 * v] != s) continue;
      const int k = slot++;
      const double* oc = a.obs_const + 8 * v;
      double* rs = a.stats + ((size_t)m * a.V + v) * SIMPLYP_NSTAT;
      const double* src = (sacc != nullptr && k < STAT_SLOTS) ? sacc + RS_COUNT * k : rs;
      const double n = src[RS_N], sse = src[RS_SSE], ssel = src[RS_SSE_LOG], ll = src[RS_LL];
      const double s1 = src[RS_S1], s2 = src[RS_S2], sos = src[RS_SOS], sabs = src[RS_SABS], shift = src[RS_SHIFT];
      const double ss_o = oc[OC_SS], ss_lo = oc[OC_SS_LOG], sum_o = oc[OC_SUM], std_o = oc[OC_STD];
      const double var_s = s2 - s1 * s1 / n;
      rs[SIMPLYP_ST_N] = n;
      rs[SIMPLYP_ST_NSE] = 1.0 - sse / ss_o;
      rs[SIMPLYP_ST_LOG_NSE] = 1.0 - ssel / ss_lo;
      rs[SIMPLYP_ST_LOGLIK] = (ll == ll) ? ll : -INFINITY;       // NaN -> -inf, MCMC.ipynb:238-240
      rs[SIMPLYP_ST_R2] = (sos * sos) / (ss_o * var_s);
      rs[SIMPLYP_ST_PBIAS] = 100.0 * (s1 + n * shift - sum_o) / sum_o;
      rs[SIMPLYP_ST_NRMSD] = 100.0 * (sabs / n) / std_o;
      rs[SIMPLYP_ST_SSE] = sse;
      rs[SIMPLYP_ST_SPEARMAN] = NAN;            // filled by spearman_kernel when rank statistics are on
      rs[SIMPLYP_ST_RESERVED] = 0.0;
      // fused all-gather: the same ten numbers into the other ranks' buffers (peer stores over NVLink; `rs` is this
      // rank's own buffer).  They are complete for the peers once this rank's flag kernel has run.
      for (int r = 0; r < a.n_peers; ++r) {
        if (r == a.my_rank) continue;
        double* dst = a.peer_stats[r] + ((size_t)(a.member_offset + m) * a.V + v) * SIMPLYP_NSTAT;
#pragma unroll
        for (int i = 0; i < SIMPLYP_NSTAT; ++i) dst[i] = rs[i];
      }
    }
  }
};

// ------------------------------------------------------------------------------------------ K1 (quad form)
// One QUAD of lanes per (member, sub-catchment) item, 8 items per warp in day lock-step (simplyp_quad.cuh).
// Shared memory: one QuadMem per quad, then the forcing ring.
// MINB = resident blocks per SM the register allocation is made for, chosen by launch_config (simplyp_plan.cuh): 2 (186
// registers), 3 (164 registers, no spills either) or 4 (128 registers, 16 warps per SM, ~150 B of spills); networks
// (STIFF) 2 (226 registers) or 3 (168 registers, 40 B of spills).
// A launch is either an ensemble of one sub-catchment (optionally the pilot or the continuation of one, optionally
// planned) or a network (tickets in dispatch order, optionally swept in epochs: KArgs::epoch_days).
enum { MODE_RUN = 0, MODE_CAL = 1 };
// Thread 0 of a block claims a list (see the PLAN_* comment) and returns its first virtual block.
__device__ int plan_claim(const KArgs& a) {
  int* plan = a.plan;
  const int nSM = a.shape.n_sm;
  unsigned smid;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
  smid &= (PLAN_MAX_SM - 1);
  const int slot = atomicAdd(plan + PLAN_SM_ARR + smid, 1);
  int* claimed = plan + PLAN_CLAIMED;
  int list = -1;
  if (slot == 0) {
    const int t = atomicAdd(plan + PLAN_FIRST_NEXT, 1);
    if (t < nSM && atomicCAS(claimed + t, 0, 1) == 0) list = t;
    __threadfence();
    atomicExch(plan + PLAN_SM_LIST + smid, list >= 0 ? list + 1 : -1);
  } else if (slot < a.shape.resident) {             // second (third) block on the SM: the list that belongs to the first
    int v = 0;
    const long long t0 = clock64();
    do {
      asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(plan + PLAN_SM_LIST + smid) : "memory");
    } while (v == 0 && clock64() - t0 < (1ll << 20));
    const int cand = slot * nSM + v - 1;
    if (v > 0 && plan_list_head(a.shape, cand) >= 0 && atomicCAS(claimed + cand, 0, 1) == 0) list = cand;
  }
  if (list < 0) {
    // no list of its own.  A launch with more blocks than lists (3 resident blocks per SM) lets that many blocks go;
    // any further block — and every block of an exact launch — takes the last list still free, so that every list is
    // claimed exactly once whatever the hardware does.
    const int spare = a.shape.n_launch() - a.shape.n_lists();
    if (spare > 0 && atomicAdd(plan + PLAN_SKIPS, 1) < spare) return -1;
    for (int l = a.shape.resident * nSM - 1; list < 0 && l >= 0; --l)
      if (plan_list_head(a.shape, l) >= 0 && atomicCAS(claimed + l, 0, 1) == 0) list = l;
  }
  return list < 0 ? -1 : plan_list_head(a.shape, list);
}

template <int MODE, int MINB, bool STIFF>
__global__ void __launch_bounds__(128, MINB) simplyp_quad_kernel(const KArgs a) {
  extern __shared__ __align__(16) double smem_cold[];
  __shared__ int s_vblock, s_epoch;
  __shared__ double s_exp2tab[EXP_TAB];
  // the placement plan exists for the 2- and 3-blocks-per-SM builds of an ensemble of one sub-catchment only
  constexpr bool PLAN = (MINB == 2 || MINB == 3) && !STIFF;
  if (threadIdx.x < EXP_TAB) s_exp2tab[threadIdx.x] = kExp2Tab[threadIdx.x];
  int vblock = (int)blockIdx.x;
  int epoch = 0, day_begin = a.day_begin, day_end = a.day_end;    // (per block in an epoch sweep of a network)
#ifdef SP_TIMELINE
  unsigned long long sp_timeline_t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(sp_timeline_t0));
#endif
  if (PLAN && a.plan != nullptr) {
    if (threadIdx.x == 0) s_vblock = plan_claim(a);
    __syncthreads();
    vblock = s_vblock;
    if (vblock < 0) return;
  } else if (STIFF && a.ticket != nullptr) {
    if (threadIdx.x == 0) {
      unsigned unit = atomicAdd(reinterpret_cast<unsigned*>(a.ticket), 1u);
      unsigned ep = 0;
      if (a.n_epochs > 1) {                         // units in epoch-major order; the item count is device-side
        // (blocks of 128 threads = 32 quads: a shift, not a 64-bit division — its subroutine's divergent slow path
        // costs the step loop its convergence proof, see IOBase)
        const unsigned n_vb = (unsigned)((a.level_item_off[a.n_levels] + 31) >> 5);
        ep = unit / n_vb;
        unit -= ep * n_vb;
      }
      s_vblock = (int)unit;
      s_epoch = (int)ep;
    }
    __syncthreads();
    vblock = s_vblock;
    if (a.n_epochs > 1) {
      // (through a warp reduction: its result is provably warp-uniform, a value read from shared memory is not — and
      // the hand-over branches of run_quad, which hold quad shuffles, depend on it; see IOBase on convergence)
      epoch = __reduce_max_sync(0xffffffffu, s_epoch);
      if (epoch >= a.n_epochs) return;
      day_begin = epoch * a.epoch_days;
      day_end = day_begin + a.epoch_days < a.day_end ? day_begin + a.epoch_days : a.day_end;
    }
  }
  const int quads_per_block = blockDim.x >> 2;
  QuadMem* qmem = reinterpret_cast<QuadMem*>(smem_cold);
  ForcingRing* ring = reinterpret_cast<ForcingRing*>(smem_cold + (size_t)quads_per_block * (sizeof(QuadMem) / sizeof(double)));
  for (;;) {                                       // one pass per virtual block of a claimed list (else one pass)
    // Networks: the item count (levels padded to whole warps) is known on the device only (stiff_group_kernel); the
    // grid is sized from a host-side upper bound, so trailing warps — and whole blocks — may have nothing to do.
    // They leave before the forcing ring counts them as consumers (a warp is either all in range or all out of it).
    int n_warps = blockDim.x >> 5;
    if (STIFF && a.level_item_off != nullptr) {
      const long long rest = a.level_item_off[a.n_levels] - (long long)vblock * quads_per_block;
      if (rest <= 0) return;
      if (rest < (long long)quads_per_block) n_warps = (int)((rest + 7) >> 3);
    }
    if (threadIdx.x == 0) {
      ring->n_consumers = (unsigned)n_warps;        // the warps of the block that integrate something
      ring->first_tile = day_begin / FORC_TILE;
      ring->end_day = day_end;
      for (int i = 0; i < FORC_SLOTS; ++i) { mbar_init(&ring->full[i], 1); ring->left[i] = 0; }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      for (int i = 0; i < FORC_SLOTS; ++i)
        if ((ring->first_tile + i) * FORC_TILE < day_end) tma_load_tile(ring, i, a.forcing, ring->first_tile + i, a.D);
    }
    __syncthreads();
    if ((int)(threadIdx.x >> 5) >= n_warps) return;  // (network launches have no further block-wide barrier)

    long long idx = (long long)vblock * quads_per_block + (threadIdx.x >> 2);
    bool valid;
    int w, m;
    if (!STIFF || a.level_item_off == nullptr) {     // one sub-catchment: items are the members
      valid = idx < a.M;
      if (!valid) idx = a.M - 1;                     // padding quads shadow the last item and write nothing
      w = 0;
      m = a.perm ? a.perm[idx] : (int)idx;
    } else {
      // group with level_item_off[lo] <= idx < level_item_off[lo+1]: bisection with a warp-uniform trip count and
      // selects instead of branches (once lo + 1 == hi the midpoint is lo itself and nothing moves any more)
      int lo = 0, hi = a.n_levels;
      for (int span = a.n_levels; span > 1; span = (span + 1) >> 1) {
        const int mid = (lo + hi) >> 1;
        const bool right = a.level_item_off[mid] <= idx;
        lo = right ? mid : lo;
        hi = right ? hi : mid;
      }
      long long local = idx - a.level_item_off[lo];
      const int o0 = a.level_order_off[lo];
      const long long n_real = (long long)(a.level_order_off[lo + 1] - o0) * a.M;
      valid = local < n_real;
      local = valid ? local : n_real - 1;
      // local = wl * M + m without a 64-bit integer division (a subroutine call with a divergent slow path: the other
      // construct that cost the step loop its convergence proof): the quotient from a double product — exact to
      // within one, local < 2^53 — then one correction step with selects
      int wl = (int)(((double)local + 0.5) * sp_rcp((double)a.M));
      long long rem = local - (long long)wl * a.M;
      wl += (rem >= a.M) ? 1 : ((rem < 0) ? -1 : 0);
      rem = local - (long long)wl * a.M;
      w = o0 + wl;
      m = (int)rem;
    }
    const int s = a.work_sc ? a.work_sc[w] : w;

    const double* mp = a.member_params + (size_t)m * SIMPLYP_NP_MEMBER;
    const double* scp = a.sc_params + (size_t)(a.Msc > 1 ? m : 0) * a.S * SIMPLYP_NP_SC;
    const double* sp = scp + (size_t)s * SIMPLYP_NP_SC;
    const double A_qr0 = scp[(size_t)a.sc_qr0 * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
    const double* spl = scp + (size_t)(a.S - 1) * SIMPLYP_NP_SC;
    const double fNCA_last = spl[SIMPLYP_SC_F_AR] * spl[SIMPLYP_SC_F_NC_AR] + spl[SIMPLYP_SC_F_NC_IG] * spl[SIMPLYP_SC_F_IG];
    const int nc_last = fNCA_last > 0.0 ? 1 : (spl[SIMPLYP_SC_F_NC_S] > 0.0 ? 2 : 0);

    // calibration: shared-memory accumulators of the fit statistics, behind the forcing ring
    // hand-over of the midnight state: pilot -> main launch of an ensemble (indexed by member), epoch -> epoch of a
    // network sweep (indexed by item)
    const bool sweep = STIFF && a.n_epochs > 1;
    const size_t ci = sweep ? (size_t)m * a.S + s : (size_t)m;
    const bool resume = sweep ? __any_sync(0xffffffffu, epoch > 0) : (a.carry != nullptr && !a.pilot_pass);
    const bool hand_over = sweep ? __any_sync(0xffffffffu, epoch + 1 < a.n_epochs) : a.pilot_pass != 0;
    const QuadCarry* cin = resume ? a.carry + ci : nullptr;
    QuadCarry* cout = hand_over ? a.carry + ci : nullptr;
    int sweep_status = 0;
    if (sweep) {                                       // the item's previous epoch (an earlier ticket) has stored its state?
      // (same shape as IOBase::wait: every condition a warp vote, so that the warp is provably converged afterwards)
      const long long t0 = clock64();
      const int* flag = a.epoch_done + ci;
      bool ok = true;
      unsigned ns = 64;
      while (ok && !__all_sync(0xffffffffu, ld_acquire_s32(flag) >= epoch)) {
        __nanosleep(ns);
        if (ns < 4096) ns *= 2;
        ok = __all_sync(0xffffffffu, (clock64() - t0) < (1ll << 37));
      }
      if (!ok) sweep_status = 4;
    }
    double* sacc = nullptr;
    if (MODE == MODE_CAL) {
      sacc = reinterpret_cast<double*>(ring + 1) + (size_t)(threadIdx.x >> 2) * STAT_STRIDE;
      if ((threadIdx.x & 3) == 0) {
        const double* src = resume ? a.carry_stats + ci * (STAT_SLOTS * RS_COUNT) : nullptr;
        // (in pairs: the 2- and 3-blocks-per-SM builds then keep the register allocation they had with 8 sums a series)
        for (int i = 0; i < STAT_SLOTS * RS_COUNT; i += 2) { sacc[i] = src ? src[i] : 0.0; sacc[i + 1] = src ? src[i + 1] : 0.0; }
      }
      __syncwarp();
    }
    QuadDev q;
    q.ql = threadIdx.x & 3;
    q.tab = s_exp2tab;
    QuadMem& qm = qmem[threadIdx.x >> 2];
    ThreadCounters cnt;
    if (MODE == MODE_CAL) {
      CalIO<STIFF> io(a, m, s, ring, mp[SIMPLYP_P_F_TDP], sacc);
      run_quad<STIFF>(q, mp, sp, A_qr0, nc_last, a.topt, day_end, valid, qm, io, cnt, day_begin, cin, cout, resume, hand_over);
      if (valid && q.ql == 0) {
        if (hand_over) {
          double* dst = a.carry_stats + ci * (STAT_SLOTS * RS_COUNT);
          for (int i = 0; i < STAT_SLOTS * RS_COUNT; ++i) dst[i] = sacc[i];
        } else {
          io.finalise();
        }
      }
      cnt.status |= io.wait_status;
    } else {
      RunIO<STIFF> io(a, m, s, ring);
      run_quad<STIFF>(q, mp, sp, A_qr0, nc_last, a.topt, day_end, valid, qm, io, cnt, day_begin, cin, cout, resume, hand_over);
      cnt.status |= io.wait_status;
    }
    if (sweep) {
      cnt.status |= sweep_status;
      if (hand_over) {                                 // state (and statistic sums) stored by this thread: publish the epoch
        if (valid && q.ql == 0) {
          // a status bit raised in this epoch travels with the state (run_quad stored its own before the waits' bits)
          if (cnt.status) a.carry[ci].status |= (int)cnt.status;
          asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(a.epoch_done + ci), "r"(epoch + 1) : "memory");
          if (a.epoch_flags_host != nullptr) {         // last item of the epoch: its rows may leave for the host now
            __threadfence();
            if (atomicAdd(a.epoch_count + epoch, 1u) + 1u == (unsigned)a.M * (unsigned)a.S) {
              __threadfence_system();
              *reinterpret_cast<volatile int*>(a.epoch_flags_host + epoch) = 1;
            }
          }
        }
        return;
      }
    }
    if (a.pilot_pass) {                                // the pilot's product: the cost of every member
      if (valid && q.ql == 0) {
        const unsigned c = (unsigned)cnt.steps;
        a.cost[m] = c;
        atomicAdd(&a.hist[c < COST_BUCKETS ? c : COST_BUCKETS - 1], 1u);
      }
      return;
    }
    if (a.diag && valid && q.ql == 0) {
      long long* dg = a.diag + ((size_t)m * a.S + s) * SIMPLYP_NDIAG;
      dg[SIMPLYP_DG_STEPS] = cnt.steps;
      dg[SIMPLYP_DG_REJECTED] = cnt.rejected;
      dg[SIMPLYP_DG_RHS] = cnt.rhs_evals;
      dg[SIMPLYP_DG_STATUS] = cnt.status;
#ifdef SP_TIMELINE                                  // analysis builds (scripts/exp_timeline.py): when and where the warp ran
      unsigned long long t1; unsigned smid;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      dg[SIMPLYP_DG_REJECTED] = (long long)sp_timeline_t0;
      dg[SIMPLYP_DG_RHS] = (long long)t1;
      dg[SIMPLYP_DG_STATUS] = (long long)smid | ((long long)vblock << 16) | ((long long)(threadIdx.x >> 5) << 40) |
                              ((long long)cnt.rejected << 44);      // cnt.rejected holds the warp's lock-step attempts here
#endif
    }
    if (!(PLAN && a.plan != nullptr)) break;
    // next virtual block of the list: every warp has left the forcing ring and the shared-memory state of its quads
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int i = 0; i < FORC_SLOTS; ++i) mbar_inval(&ring->full[i]);
      s_vblock = plan_list_next(a.shape, vblock);
    }
    __syncthreads();
    vblock = s_vblock;
    if (vblock < 0) break;
#ifdef SP_TIMELINE
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(sp_timeline_t0));
#endif
  }
}

// ------------------------------------------------------------------------------------------ rank statistics
// Spearman's r (visualise_results.py:444-445: pandas corr(method='spearman') = Pearson correlation of average
// ranks).  The observation ranks are shared by all members: one block per series ranks them once
// (obs_rank[v][d], NaN where there is no observation) and stores the sum of squares about the mean rank.
__global__ void obs_rank_kernel(const double* obs, int D, double* obs_rank, double* obs_const) {
  const int v = blockIdx.x;
  const double* o = obs + (size_t)v * D;
  double* rk = obs_rank + (size_t)v * D;
  __shared__ double red[256];
  const double n = obs_const[8 * v + OC_N];
  const double mean_rank = 0.5 * (n + 1.0);
  double ss = 0.0;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const double x = o[d];
    double r = NAN;
    if (x == x) {
      int less = 0, equal = 0;
      for (int j = 0; j < D; ++j) { const double y = o[j]; less += (y < x); equal += (y == x); }
      r = less + 0.5 * (equal + 1);                 // average rank of a tie group
      ss += (r - mean_rank) * (r - mean_rank);
    }
    rk[d] = r;
  }
  red[threadIdx.x] = ss;
  __syncthreads();
  for (int k = blockDim.x / 2; k > 0; k >>= 1) {
    if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k];
    __syncthreads();
  }
  if (threadIdx.x == 0) obs_const[8 * v + OC_SS_RANK] = red[0];
}

// One block per (member, series): the simulated values of the observed days are compacted into shared memory
// together with the observation ranks, ranked by counting (ties share the mean rank) and correlated.
// Dynamic shared memory: 2 * cap doubles, cap >= D (longer records: spearman_long_kernel).
__global__ void spearman_kernel(const double* sim_obs, const double* obs_rank, const double* obs_const, int V, int D,
                                int cap, double* stats) {
  extern __shared__ double sh[];
  double* s_sim = sh;
  double* s_rk = sh + cap;
  __shared__ int s_n;
  __shared__ double red[2][128];
  const int mv = blockIdx.x, v = mv % V;
  const double* sim = sim_obs + (size_t)mv * D;
  const double* rk = obs_rank + (size_t)v * D;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const double r = rk[d];
    if (r == r) {
      const double x = sim[d];
      if (x == x) {                                 // pairs with a NaN on either side are dropped (:435-436)
        const int k = atomicAdd(&s_n, 1);
        if (k < cap) { s_sim[k] = x; s_rk[k] = r; }
      }
    }
  }
  __syncthreads();
  const int n = s_n;
  double* out = stats + (size_t)mv * SIMPLYP_NSTAT + SIMPLYP_ST_SPEARMAN;
  if (n > cap || n < 2) { if (threadIdx.x == 0) *out = NAN; return; }
  // a NaN simulated value changes the set of pairs: the observation ranks must then be recomputed among the
  // pairs kept (pandas ranks after dropna) — rare (a failed member); detected by comparing n with the series' n
  const bool rerank_obs = (double)n != obs_const[8 * v + OC_N];
  const double mean_rank = 0.5 * (n + 1.0);
  double sxy = 0.0, sxx = 0.0, syy = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double x = s_sim[i];
    int less = 0, equal = 0;
    for (int j = 0; j < n; ++j) { const double y = s_sim[j]; less += (y < x); equal += (y == x); }
    const double rs = less + 0.5 * (equal + 1);
    double ro = s_rk[i];
    if (rerank_obs) {
      int l2 = 0, e2 = 0;
      for (int j = 0; j < n; ++j) { const double y = s_rk[j]; l2 += (y < ro); e2 += (y == ro); }
      ro = l2 + 0.5 * (e2 + 1);
      syy += (ro - mean_rank) * (ro - mean_rank);
    }
    sxy += (rs - mean_rank) * (ro - mean_rank);
    sxx += (rs - mean_rank) * (rs - mean_rank);
  }
  red[0][threadIdx.x] = sxy; red[1][threadIdx.x] = sxx;
  __syncthreads();
  for (int k = blockDim.x / 2; k > 0; k >>= 1) {
    if (threadIdx.x < k) { red[0][threadIdx.x] += red[0][threadIdx.x + k]; red[1][threadIdx.x] += red[1][threadIdx.x + k]; }
    __syncthreads();
  }
  const double cxy = red[0][0], cxx = red[1][0];
  __syncthreads();
  if (rerank_obs) {
    red[0][threadIdx.x] = syy;
    __syncthreads();
    for (int k = blockDim.x / 2; k > 0; k >>= 1) {
      if (threadIdx.x < k) red[0][threadIdx.x] += red[0][threadIdx.x + k];
      __syncthreads();
    }
  }
  if (threadIdx.x == 0) {
    const double cyy = rerank_obs ? red[0][0] : obs_const[8 * v + OC_SS_RANK];
    *out = cxy / sqrt(cxx * cyy);
  }
}

// The same for series too long for shared memory (more than ~12,800 days, i.e. 35 years of daily observations): no
// compaction; every thread ranks its days by counting over the whole series in global memory (L1/L2 resident:
// 16 B per day).  O(n D) reads per (member, series) — slower, but rare and exact.
__global__ void spearman_long_kernel(const double* sim_obs, const double* obs_rank, const double* obs_const, int V, int D,
                                     double* stats) {
  __shared__ double red[3][128];
  __shared__ int s_cnt[128];
  const int mv = blockIdx.x, v = mv % V;
  const double* sim = sim_obs + (size_t)mv * D;
  const double* rk = obs_rank + (size_t)v * D;
  int cnt = 0;
  for (int d = threadIdx.x; d < D; d += blockDim.x) cnt += (rk[d] == rk[d]) && (sim[d] == sim[d]);
  s_cnt[threadIdx.x] = cnt;
  __syncthreads();
  for (int k = blockDim.x / 2; k > 0; k >>= 1) {
    if (threadIdx.x < k) s_cnt[threadIdx.x] += s_cnt[threadIdx.x + k];
    __syncthreads();
  }
  const int n = s_cnt[0];
  double* out = stats + (size_t)mv * SIMPLYP_NSTAT + SIMPLYP_ST_SPEARMAN;
  if (n < 2) { if (threadIdx.x == 0) *out = NAN; return; }
  const bool rerank_obs = (double)n != obs_const[8 * v + OC_N];     // see spearman_kernel
  const double mean_rank = 0.5 * (n + 1.0);
  double sxy = 0.0, sxx = 0.0, syy = 0.0;
  for (int i = threadIdx.x; i < D; i += blockDim.x) {
    const double x = sim[i];
    double ro = rk[i];
    if (!(x == x) || !(ro == ro)) continue;
    int less = 0, equal = 0, l2 = 0, e2 = 0;
    for (int j = 0; j < D; ++j) {
      const double y = sim[j], r = rk[j];
      const bool ok = (y == y) && (r == r);
      less += ok && (y < x); equal += ok && (y == x);
      if (rerank_obs) { l2 += ok && (r < ro); e2 += ok && (r == ro); }
    }
    const double rs = less + 0.5 * (equal + 1);
    if (rerank_obs) ro = l2 + 0.5 * (e2 + 1);
    sxy += (rs - mean_rank) * (ro - mean_rank);
    sxx += (rs - mean_rank) * (rs - mean_rank);
    syy += (ro - mean_rank) * (ro - mean_rank);
  }
  red[0][threadIdx.x] = sxy; red[1][threadIdx.x] = sxx; red[2][threadIdx.x] = syy;
  __syncthreads();
  for (int k = blockDim.x / 2; k > 0; k >>= 1) {
    if (threadIdx.x < k) for (int j = 0; j < 3; ++j) red[j][threadIdx.x] += red[j][threadIdx.x + k];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = red[0][0] / sqrt(red[1][0] * (rerank_obs ? red[2][0] : obs_const[8 * v + OC_SS_RANK]));
}

// ------------------------------------------------------------------------------------------ waterbody sums
// sum_to_waterbody (model.py:851-900) on the raw output: for every (member, day) the reaches flagged
// In_final_flux? == 1 are summed — Q_cumecs (= Qr*A_catch*1000/86400, :784), Msus/TDP/PP daily fluxes — and the
// concentrations (:889-892) and derived species (derived_P_species, :831-847) follow.  One thread per (member, day);
// consecutive threads take consecutive days, so the strided row reads of a warp fall in neighbouring rows.
// wb[m][d][SIMPLYP_NWB] = Q_cumecs, Msus_kg/day, TDP_kg/day, PP_kg/day, SS_mgl, TDP_mgl, PP_mgl, TP_mgl,
//                          TP_kg/day, SRP_mgl, SRP_kg/day
__global__ void waterbody_kernel(const double* out, const double* sc_params, const double* member_params,
                                 const int* reaches, int n_reaches, int M, int S, int D, int Msc, double* wb) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)M * D) return;
  const int m = (int)(idx / D), d = (int)(idx - (long long)m * D);
  const double* scp = sc_params + (size_t)(Msc > 1 ? m : 0) * S * SIMPLYP_NP_SC;
  double q = 0.0, ms = 0.0, td = 0.0, pp = 0.0;
  for (int k = 0; k < n_reaches; ++k) {
    const int s = reaches[k];
    const double* row = out + (((size_t)m * S + s) * D + d) * SIMPLYP_NOUT;
    q += row[SIMPLYP_O_QR] * scp[(size_t)s * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH] * 1000.0 / 86400.0;
    ms += row[SIMPLYP_O_MSUS_FLUX];
    td += row[SIMPLYP_O_TDP_FLUX];
    pp += row[SIMPLYP_O_PP_FLUX];
  }
  const double f_TDP = member_params[(size_t)m * SIMPLYP_NP_MEMBER + SIMPLYP_P_F_TDP];
  const double c = 1000.0 / 86400.0;
  double* w = wb + (size_t)idx * SIMPLYP_NWB;
  const double ss_mgl = (ms / q) * c, tdp_mgl = (td / q) * c, pp_mgl = (pp / q) * c;
  w[0] = q; w[1] = ms; w[2] = td; w[3] = pp; w[4] = ss_mgl; w[5] = tdp_mgl; w[6] = pp_mgl;
  w[7] = tdp_mgl + pp_mgl;        // TP_mgl   (:842)
  w[8] = td + pp;                 // TP_kg/day (:843)
  w[9] = tdp_mgl * f_TDP;         // SRP_mgl  (:844)
  w[10] = td * f_TDP;             // SRP_kg/day (:845)
}

// ------------------------------------------------------------------------------------------ Thornthwaite PET
// daily_PET (inputs.py:232-312) for a record of whole calendar years, one block: monthly mean daylight hours from the
// latitude (:416-445; FAO-56 eq. 24, 25, 34 at :370-414), monthly mean air temperature, Thornthwaite's monthly PET per
// year (:447-508), divided by the days of the month, placed on the 16th and interpolated linearly to the days (the
// days before the first and after the last 16th take that value, as pandas' limit_direction='both' does).
// Dynamic shared memory: 2 * n_months doubles.
__global__ void thornthwaite_kernel(int D, int NM, const double* t_air, int t_stride, const int* month_start,
                                    const int* year_is_leap, double lat_rad, double* pet, int pet_stride) {
  extern __shared__ double sh_pet[];
  double* s_tmean = sh_pet;            // [NM] monthly mean air temperature, negative values counted as zero
  double* s_pet = sh_pet + NM;         // [NM] PET per day of the month (value on the 16th)
  __shared__ double s_dlh[2][12];
  const int mdays[12] = {31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31};
  if (threadIdx.x < 24) {
    const int leap = threadIdx.x / 12, mon = threadIdx.x % 12;
    int doy = 1;
    for (int k = 0; k < mon; ++k) doy += mdays[k] + ((leap && k == 1) ? 1 : 0);
    const int n = mdays[mon] + ((leap && mon == 1) ? 1 : 0);
    double total = 0.0;
    for (int k = 0; k < n; ++k, ++doy) {
      const double sd = 0.409 * sin((2.0 * M_PI / 365.0) * doy - 1.39);
      const double c = -tan(lat_rad) * tan(sd);
      total += (24.0 / M_PI) * acos(fmin(fmax(c, -1.0), 1.0));
    }
    s_dlh[leap][mon] = total / n;
  }
  for (int m = threadIdx.x; m < NM; m += blockDim.x) {
    const int d0 = month_start[m], d1 = month_start[m + 1];
    double sum = 0.0;
    for (int d = d0; d < d1; ++d) sum += t_air[(size_t)d * t_stride];
    const double t = sum / (d1 - d0);
    s_tmean[m] = t >= 0.0 ? t : 0.0;
  }
  __syncthreads();
  for (int m = threadIdx.x; m < NM; m += blockDim.x) {
    // bit 0: the year is a leap year (days of February); bit 1: the year takes the leap-year daylight table — the
    // reference keeps that table for every year AFTER its first leap year too (inputs.py:269-273 overwrites the
    // variable the non-leap branch reads), so the host sets bit 1 accordingly under strict quirks
    const int y = m / 12, mon = m % 12, leap = year_is_leap[y] & 1, dl = (year_is_leap[y] >> 1) & 1;
    double heat = 0.0;
    for (int k = 0; k < 12; ++k) {
      const double x = s_tmean[12 * y + k] / 5.0;
      if (x > 0.0) heat += pow(x, 1.514);
    }
    const double a = (6.75e-07 * pow(heat, 3.0)) - (7.71e-05 * pow(heat, 2.0)) + (1.792e-02 * heat) + 0.49239;
    const double N = mdays[mon] + ((leap && mon == 1) ? 1 : 0);
    const double ta = s_tmean[m];
    s_pet[m] = (1.6 * (s_dlh[dl][mon] / 12.0) * (N / 30.0) * pow(10.0 * ta / heat, a) * 10.0) / N;
  }
  __syncthreads();
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    int lo = 0, hi = NM;                            // month with month_start[lo] <= d < month_start[lo+1]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (month_start[mid] <= d) lo = mid; else hi = mid;
    }
    const int m0 = (d >= month_start[lo] + 15) ? lo : lo - 1, m1 = m0 + 1;
    double v;
    if (m0 < 0) v = s_pet[0];
    else if (m1 >= NM) v = s_pet[NM - 1];
    else {
      const int x0 = month_start[m0] + 15, x1 = month_start[m1] + 15;
      const double slope = (s_pet[m1] - s_pet[m0]) / (double)(x1 - x0);
      v = slope * (double)(d - x0) + s_pet[m0];
    }
    pet[(size_t)d * pet_stride] = v;
  }
}

// ------------------------------------------------------------------------------------------ cost ordering
// Counting sort of the members by pilot cost, heaviest first: hist[] -> start offsets (one block), then scatter.
__global__ void cost_scan_kernel(unsigned* hist) {
  __shared__ unsigned part[1024];
  constexpr int PER = COST_BUCKETS / 1024;
  // thread t owns buckets [PER*t, PER*t+PER) counted from the TOP (descending cost)
  unsigned loc[PER], sum = 0;
#pragma unroll
  for (int k = 0; k < PER; ++k) { loc[k] = hist[COST_BUCKETS - 1 - (PER * threadIdx.x + k)]; sum += loc[k]; }
  part[threadIdx.x] = sum;
  __syncthreads();
  for (int d = 1; d < 1024; d <<= 1) {            // inclusive Hillis-Steele scan
    const unsigned v = threadIdx.x >= d ? part[threadIdx.x - d] : 0u;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  unsigned run = part[threadIdx.x] - sum;         // exclusive prefix of this thread's first bucket
#pragma unroll
  for (int k = 0; k < PER; ++k) { hist[COST_BUCKETS - 1 - (PER * threadIdx.x + k)] = run; run += loc[k]; }
}
// Scatter of the members into their places: rank by the counting sort (heaviest first), place by the member layout
// of the plan (simplyp_plan.cuh; the identity for an unplanned launch).
__global__ void cost_scatter_kernel(const unsigned* cost, unsigned* offsets, int* perm, int M, MemberLayout L) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const unsigned c = cost[m];
  const int rank = (int)atomicAdd(&offsets[c < COST_BUCKETS ? c : COST_BUCKETS - 1], 1u);
  perm[member_layout_index(rank, L)] = m;
}

// ------------------------------------------------------------------------------------------ obs constants
// One block per observed series: n, mean, sum of squares about the mean (plain and log), sum, std.
__global__ void obs_const_kernel(const double* obs, int D, double* obs_const, double* obs_log) {
  const int v = blockIdx.x;
  const double* o = obs + (size_t)v * D;
  for (int d = threadIdx.x; d < D; d += blockDim.x) obs_log[(size_t)v * D + d] = log(o[d]);   // NaN stays NaN
  __shared__ double red[5][256];
  double n = 0, s = 0, sl = 0;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const double x = o[d];
    if (x == x) { n += 1.0; s += x; sl += log(x); }
  }
  red[0][threadIdx.x] = n; red[1][threadIdx.x] = s; red[2][threadIdx.x] = sl;
  __syncthreads();
  for (int k = blockDim.x / 2; k > 0; k >>= 1) {
    if (threadIdx.x < k) for (int j = 0; j < 3; ++j) red[j][threadIdx.x] += red[j][threadIdx.x + k];
    __syncthreads();
  }
  const double N = red[0][0], mean = red[1][0] / N, meanl = red[2][0] / N, sum = red[1][0];
  __syncthreads();
  double ss = 0, ssl = 0;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const double x = o[d];
    if (x == x) { ss += (x - mean) * (x - mean); const double l = log(x) - meanl; ssl += l * l; }
  }
  red[3][threadIdx.x] = ss; red[4][threadIdx.x] = ssl;
  __syncthreads();
  for (int k = blockDim.x / 2; k > 0; k >>= 1) {
    if (threadIdx.x < k) for (int j = 3; j < 5; ++j) red[j][threadIdx.x] += red[j][threadIdx.x + k];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double* oc = obs_const + 8 * v;
    oc[OC_N] = N; oc[OC_MEAN] = mean; oc[OC_SS] = red[3][0]; oc[OC_MEAN_LOG] = meanl;
    oc[OC_SS_LOG] = red[4][0]; oc[OC_SUM] = sum; oc[OC_STD] = sqrt(red[3][0] / N); oc[7] = 0.0;
  }
}

// ------------------------------------------------------------------------------------------ FP64 peak probe
__global__ void fp64_peak_kernel(double* sink, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
      x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
  }
  const double r = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (r == 123.456) sink[0] = r;
}

// one warp, one dependent DFMA chain: cycles per dependent DFMA = the fp64 pipe latency
__global__ void fp64_latency_kernel(double* sink, long long* cycles, int iters, double a, double b) {
  double x = threadIdx.x;
  const long long t0 = clock64();
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 16; ++u) x = fma(x, a, b);
  }
  const long long t1 = clock64();
  if (threadIdx.x == 0) cycles[0] = t1 - t0;
  if (x == 123.456) sink[0] = x;
}

// ------------------------------------------------------------------------------------------ fused all-gather: flags
// After the integration kernel of a rank (same stream): raise `step` in every peer's flag array, then wait until every
// peer has raised it here.  The integration kernel has completed, so its peer stores are performed; the system-scope
// fence + release order them before the flag for the peer that acquires it.  One thread per peer; a peer that does
// not answer within ~2 s (globaltimer) sets status bit 8 instead of hanging the device.
struct PeerFlags { int* bufs[SIMPLYP_MAX_RANKS]; };
__global__ void peer_flag_kernel(PeerFlags f, int n, int rank, int step, long long* status_word) {
  const int p = threadIdx.x;
  if (p >= n || p == rank) return;
  __threadfence_system();
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(f.bufs[p] + rank), "r"(step) : "memory");
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (;;) {
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(f.bufs[rank] + p) : "memory");
    if (v - step >= 0) break;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 2000000000ull) {
      if (status_word) atomicOr(reinterpret_cast<unsigned long long*>(status_word), 8ull);
      break;
    }
    __nanosleep(200);
  }
}

// ------------------------------------------------------------------------------------------ host helpers
int topology_levels(int S, const int32_t* po, const int32_t* pid, std::vector<int>& lvl) {
  lvl.assign(S, 0);
  int nl = S > 0 ? 1 : 0;
  for (int s = 0; s < S; ++s) {
    if (po[s + 1] < po[s]) return SIMPLYP_EINVAL;
    int L = 0;
    for (int e = po[s]; e < po[s + 1]; ++e) {
      const int p = pid[e];
      if (p < 0 || p >= s) return SIMPLYP_EINVAL;   // parents must come earlier in run order
      L = L > lvl[p] + 1 ? L : lvl[p] + 1;
    }
    lvl[s] = L;
    nl = nl > L + 1 ? nl : L + 1;
  }
  return nl;
}

size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

struct WsLayout {
  size_t off_po, off_pid, off_bylevel, off_lvlstart, off_topo_end, off_order, off_area, off_lvl_items, off_lvl_order, off_oc,
      off_cost, off_hist, off_perm, off_plan, off_carry, off_carry_stats, off_ticket, off_progress, off_epoch_done,
      off_epoch_count, off_flux, off_obs_log,
      off_obs_rank, off_sim_obs, total;
};

WsLayout ws_layout(const SimplypDims& d, int n_edges, bool cal, bool ranks = false) {
  WsLayout L;
  size_t o = 0;
  // [off_po, off_topo_end): the host-built topology tables, filled by ONE copy from a pinned staging image
  L.off_po = o;    o = align_up(o + sizeof(int) * ((size_t)d.n_sc + 1));
  L.off_pid = o;   o = align_up(o + sizeof(int) * (size_t)(n_edges > 0 ? n_edges : 1));
  L.off_bylevel = o;  o = align_up(o + sizeof(int) * (size_t)d.n_sc);            // reaches sorted by (level, run order)
  L.off_lvlstart = o; o = align_up(o + sizeof(int) * ((size_t)d.n_sc + 1));      // [n_levels+1] offsets into it
  L.off_topo_end = o;
  L.off_order = o; o = align_up(o + sizeof(int) * (size_t)d.n_sc);
  L.off_area = o;  o = align_up(o + sizeof(double) * (size_t)d.n_sc);            // area upstream of (and including) a reach
  L.off_lvl_items = o; o = align_up(o + sizeof(long long) * (2 * (size_t)d.n_sc + 1));   // <= 2 groups per level
  L.off_lvl_order = o; o = align_up(o + sizeof(int) * (2 * (size_t)d.n_sc + 1));
  L.off_oc = o;    o = align_up(o + sizeof(double) * 8 * (size_t)(d.n_obs_series > 0 ? d.n_obs_series : 1));
  L.off_cost = o;  o = align_up(o + sizeof(unsigned) * (size_t)d.n_members);
  L.off_hist = o;  o = align_up(o + sizeof(unsigned) * COST_BUCKETS);
  L.off_perm = o;  o = align_up(o + sizeof(int) * (size_t)d.n_members);
  L.off_plan = o;  if (d.n_sc == 1) o = align_up(o + sizeof(int) * (size_t)PLAN_INTS);
  // midnight states handed over between launches (ensemble: pilot -> main, per member) or epochs (network: per item)
  const size_t n_carry = d.n_sc == 1 ? (d.n_members >= 512 ? (size_t)d.n_members : 0) : (size_t)d.n_members * d.n_sc;
  L.off_carry = o;
  o = align_up(o + sizeof(QuadCarry) * n_carry);
  L.off_carry_stats = o;
  if (cal) o = align_up(o + sizeof(double) * STAT_SLOTS * RS_COUNT * n_carry);
  L.off_ticket = o; o = align_up(o + sizeof(int));
  L.off_progress = o;
  if (d.n_sc > 1) o = align_up(o + sizeof(int) * (size_t)d.n_members * d.n_sc);
  L.off_epoch_done = o;
  if (d.n_sc > 1) o = align_up(o + sizeof(int) * (size_t)d.n_members * d.n_sc);
  L.off_epoch_count = o;
  if (d.n_sc > 1) o = align_up(o + sizeof(unsigned) * ((size_t)d.n_days / FORC_TILE + 2));
  L.off_flux = o;
  if (cal && d.n_sc > 1) o = align_up(o + sizeof(double) * 4 * (size_t)d.n_members * d.n_sc * d.n_days);
  L.off_obs_log = o;
  if (cal) o = align_up(o + sizeof(double) * (size_t)(d.n_obs_series > 0 ? d.n_obs_series : 1) * d.n_days);
  L.off_obs_rank = o;
  if (cal && ranks) o = align_up(o + sizeof(double) * (size_t)(d.n_obs_series > 0 ? d.n_obs_series : 1) * d.n_days);
  L.off_sim_obs = o;
  if (cal && ranks) o = align_up(o + sizeof(double) * (size_t)d.n_members * (d.n_obs_series > 0 ? d.n_obs_series : 1) * d.n_days);
  L.total = o;
  return L;
}

// Pinned host images of the topology tables of earlier calls.  The *_device entry points copy the caller's CSR
// arrays (pageable host memory the caller may free or change right after the call) into such an image and enqueue
// ONE asynchronous copy from it, so that they never synchronise and can be captured into a CUDA graph (a replay
// reads the image again: images are kept until simplyp_release_cache()).  A call whose tables equal an earlier
// image reuses it — and then allocates nothing, which stream capture in its strict mode requires.
struct TopoImage { uint64_t hash; size_t bytes; char* host; };
std::mutex g_topo_mutex;
std::vector<TopoImage> g_topo_images;

int topo_image_get(const std::vector<char>& img, const char** out) {
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < img.size(); ++i) { h ^= (unsigned char)img[i]; h *= 1099511628211ull; }
  std::lock_guard<std::mutex> lock(g_topo_mutex);
  for (const TopoImage& t : g_topo_images)
    if (t.hash == h && t.bytes == img.size() && memcmp(t.host, img.data(), img.size()) == 0) { *out = t.host; return SIMPLYP_OK; }
  char* host = nullptr;
  SP_CUDA(cudaMallocHost(&host, img.size()));
  memcpy(host, img.data(), img.size());
  g_topo_images.push_back({h, img.size(), host});
  *out = host;
  return SIMPLYP_OK;
}

int check_common(const SimplypDims* dims, const SimplypOptions* opt, const void* forcing, const void* mp,
                 const void* scp, const int32_t* po) {
  if (!dims || !opt || !forcing || !mp || !scp || !po) return fail(SIMPLYP_EINVAL, "null argument%s");
  if (dims->n_members <= 0 || dims->n_sc <= 0 || dims->n_days < 0) return fail(SIMPLYP_EINVAL, "bad dims%s");
  if (dims->n_sc_param_sets != 1 && dims->n_sc_param_sets != dims->n_members)
    return fail(SIMPLYP_EINVAL, "n_sc_param_sets must be 1 or n_members%s");
  if (opt->sc_qr0 < 0 || opt->sc_qr0 >= dims->n_sc) return fail(SIMPLYP_EINVAL, "sc_qr0 out of range%s");
  if (!(opt->rtol > 0.0) || !(opt->atol >= 0.0) || !(opt->step_len > 0.0))
    return fail(SIMPLYP_EINVAL, "rtol/atol/step_len must be positive%s");
  if (opt->lanes_per_item != 0 && opt->lanes_per_item != 4)
    return fail(SIMPLYP_EINVAL, "lanes_per_item must be 0 (default) or 4: the one-thread-per-item kernel was retired%s");
  return SIMPLYP_OK;
}

ThreadOptions make_topt(const SimplypOptions& o) {
  ThreadOptions t;
  t.rtol = o.rtol; t.atol = o.atol; t.step_len = o.step_len;
  t.max_steps_per_day = o.max_steps_per_day > 0 ? o.max_steps_per_day : 5000;
  t.dynamic_epc0 = o.dynamic_epc0; t.dynamic_erod = o.dynamic_erodibility;
  t.run_mode_cal = o.run_mode_cal; t.strict_quirks = o.strict_quirks;
  t.snow_on_device = o.snow_on_device;
  return t;
}

// The quad kernel in the register variant `minb` (launch_config).  Networks (STIFF) have no 4-blocks build.
template <int MODE, bool STIFF>
void launch_quad(int minb, long long grid, size_t smem, cudaStream_t st, const KArgs& a) {
  const unsigned g = (unsigned)grid, block = 128;
  if (minb == 2) simplyp_quad_kernel<MODE, 2, STIFF><<<g, block, smem, st>>>(a);
  else if (minb == 3 || STIFF) simplyp_quad_kernel<MODE, 3, STIFF><<<g, block, smem, st>>>(a);
  else if constexpr (!STIFF) simplyp_quad_kernel<MODE, 4, false><<<g, block, smem, st>>>(a);
}

// Pilot + counting sort: fills a.perm (one sub-catchment, quad kernel).  3 small launches + the pilot.
template <int MODE>
int order_members_by_cost(const SimplypDims& dims, const LaunchConfig& c, KArgs& a, const WsLayout& L, char* ws,
                          size_t smem, cudaStream_t st) {
  if (c.pilot_days == 0) return SIMPLYP_OK;
  // the pilot is the run's own first `pilot_days` days (same kernel, member order): it leaves every member's midnight
  // state in the carry area, and the main launch continues from there in cost order
  a.carry = reinterpret_cast<QuadCarry*>(ws + L.off_carry);
  a.carry_stats = reinterpret_cast<double*>(ws + L.off_carry_stats);
  KArgs p = a;
  p.day_end = c.pilot_days;
  p.diag = nullptr;
  p.perm = nullptr;
  p.pilot_pass = 1;
  p.cost = reinterpret_cast<unsigned*>(ws + L.off_cost);
  p.hist = reinterpret_cast<unsigned*>(ws + L.off_hist);
  a.day_begin = c.pilot_days;
  int* perm = reinterpret_cast<int*>(ws + L.off_perm);
  SP_CUDA(cudaMemsetAsync(p.hist, 0, sizeof(unsigned) * COST_BUCKETS, st));
  launch_quad<MODE, false>(c.pilot_minb, (dims.n_members + 31ll) / 32, smem, st, p);
  cost_scan_kernel<<<1, 1024, 0, st>>>(p.hist);
  MemberLayout lay = {0, 0, 0, 0};
  if (c.plan) {                                      // see PLAN_*
    lay = member_layout(c.shape, dims.n_members, c.solo);
    int* plan = reinterpret_cast<int*>(ws + L.off_plan);
    SP_CUDA(cudaMemsetAsync(plan, 0, sizeof(int) * PLAN_INTS, st));
    a.plan = plan;
    a.shape = c.shape;
  }
  cost_scatter_kernel<<<(dims.n_members + 255) / 256, 256, 0, st>>>(p.cost, p.hist, perm, dims.n_members, lay);
  g_launches.fetch_add(3);
  SP_CUDA(cudaGetLastError());
  a.perm = perm;
  return SIMPLYP_OK;
}

// Orders the reaches of every topological level for the network launch: the reaches that are expected to be stiff
// first, then the rest, so that the lock-step warps of a level hold either Rosenbrock items or explicit ones and do not
// execute both attempts per iteration.  The expectation is an estimate from the FIRST parameter set: reach rate
// constant at a nominal runoff of 3 mm/d over the whole upstream area (a_Q 86400/L (3 A_upstream/A_own)^b_Q / (1-b_Q),
// model.py:127-130) against the kernel's switching rate.  It only steers the grouping: the method itself is still
// chosen per item and day in the integration kernel.  One block; runs on the device because the parameters live
// there and the *_device entry points must not synchronise.
//   by_level[S], lvl_start[n_levels+1] : reaches sorted by (level, run order), from the host
//   order[S]                           : reaches in launch order (group by group)
//   grp_order[2 n_levels + 1]          : offsets of the groups into order[]
//   grp_items[2 n_levels + 1]          : cumulative item counts, every group padded to whole warps of 8 quads
__global__ void stiff_group_kernel(int S, int n_levels, int M, const int* by_level, const int* lvl_start, const int* po,
                                   const int* pid, const double* sc_params, const double* member_params, double* area_up,
                                   int* order, int* grp_order, long long* grp_items) {
  const double aQ = member_params[SIMPLYP_P_A_Q], bQ = member_params[SIMPLYP_P_B_Q];
  for (int L = 0; L < n_levels; ++L) {                 // parents sit on lower levels
    for (int k = lvl_start[L] + threadIdx.x; k < lvl_start[L + 1]; k += blockDim.x) {
      const int s = by_level[k];
      double a = sc_params[(size_t)s * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
      for (int e = po[s]; e < po[s + 1]; ++e) a += area_up[pid[e]];
      area_up[s] = a;
    }
    __syncthreads();
  }
  for (int L = threadIdx.x; L < n_levels; L += blockDim.x) {
    const int k0 = lvl_start[L], k1 = lvl_start[L + 1];
    int n_stiff = 0;
    for (int pass = 0; pass < 2; ++pass) {             // stable partition: stiff reaches, then the others
      int w = k0 + (pass ? n_stiff : 0);
      for (int k = k0; k < k1; ++k) {
        const int s = by_level[k];
        const double* sp = sc_params + (size_t)s * SIMPLYP_NP_SC;
        const double qr = 3.0 * area_up[s] / sp[SIMPLYP_SC_A_CATCH];
        const double rate = aQ * 86400.0 / sp[SIMPLYP_SC_L_REACH] * pow(qr, bQ) / (1.0 - bQ);
        const bool stiff = rate > SP_STIFF_RATE;
        if (stiff == (pass == 0)) { order[w++] = s; if (pass == 0) ++n_stiff; }
      }
    }
    grp_order[2 * L] = k0;
    grp_order[2 * L + 1] = k0 + n_stiff;
  }
  if (threadIdx.x == 0) grp_order[2 * n_levels] = S;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long run = 0;
    grp_items[0] = 0;
    for (int g = 0; g < 2 * n_levels; ++g) {
      const long long n_real = (long long)(grp_order[g + 1] - grp_order[g]) * M;
      run += (n_real + 7) / 8 * 8;                     // an empty group takes no items
      grp_items[g + 1] = run;
    }
  }
}

// Shared launcher: one launch; the reach DAG is swept as a day-skewed wavefront inside the kernel.  Everything is
// enqueued on `st`; nothing here waits for the device.
// What a *_host entry point needs to stream finished epochs of a network launch to the caller (see KArgs): in, the
// device pointer of its mapped flags and how many there are; out, the epochs of the launch (n_epochs <= 1: no sweep,
// nothing is signalled).
struct EpochStream {
  int* flags_dev = nullptr;
  int capacity = 0;
  int n_epochs = 0, epoch_days = 0;
};

template <bool CAL>
int launch_levels(const SimplypDims& dims, const SimplypOptions& opt, KArgs a, const int32_t* po_host,
                  const int32_t* pid_host, char* ws, cudaStream_t st, EpochStream* es = nullptr) {
  const int S = dims.n_sc;
  std::vector<int> lvl;
  const int nl = topology_levels(S, po_host, pid_host, lvl);
  if (nl < 0) return fail(SIMPLYP_EINVAL, "topology: parents must precede children in run order%s");
  const int E = po_host[S];
  const WsLayout L = ws_layout(dims, E, CAL);
  constexpr int MODE = CAL ? MODE_CAL : MODE_RUN;
  const int qpb = 32;                        // items per block of 128 threads
  const size_t smem = (size_t)qpb * sizeof(QuadMem) + sizeof(ForcingRing) +
                      (CAL ? (size_t)qpb * STAT_STRIDE * sizeof(double) : 0);
  a.n_work = S;
  int dev = 0, n_sm = 0;
  SP_CUDA(cudaGetDevice(&dev));
  SP_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  const LaunchOverrides ov = read_launch_overrides();

  if (S == 1 && E == 0) {                    // an ensemble of one sub-catchment: items are the members
    int* zp = nullptr;
    SP_CUDA(cudaGetSymbolAddress((void**)&zp, g_zero_offsets));
    a.parent_offsets = zp;   // {0, 0}: no parents
    a.parent_ids = zp;
    const LaunchConfig c =
        launch_config({dims.n_members, dims.n_days, false, 0, 0, opt.pilot_days, ws != nullptr, n_sm}, ov);
    const int rc = order_members_by_cost<MODE>(dims, c, a, L, ws, smem, st);
    if (rc) return rc;
    launch_quad<MODE, false>(c.minb, c.grid, smem, st, a);
    g_launches.fetch_add(1);
    SP_CUDA(cudaGetLastError());
    return SIMPLYP_OK;
  }

  // ---- a network: topology tables -> workspace (one copy from a pinned image), grouping on the device
  if (!ws) return fail(SIMPLYP_EINVAL, "workspace required for n_sc > 1%s");
  std::vector<char> img(L.off_topo_end - L.off_po, 0);
  int* i_po = reinterpret_cast<int*>(img.data() + (L.off_po - L.off_po));
  int* i_pid = reinterpret_cast<int*>(img.data() + (L.off_pid - L.off_po));
  int* i_byl = reinterpret_cast<int*>(img.data() + (L.off_bylevel - L.off_po));
  int* i_ls = reinterpret_cast<int*>(img.data() + (L.off_lvlstart - L.off_po));
  memcpy(i_po, po_host, sizeof(int) * (S + 1));
  if (E > 0) memcpy(i_pid, pid_host, sizeof(int) * E);
  for (int s = 0; s < S; ++s) i_ls[lvl[s] + 1] += 1;
  for (int l = 0; l < nl; ++l) i_ls[l + 1] += i_ls[l];
  {
    std::vector<int> fill(i_ls, i_ls + nl);
    for (int s = 0; s < S; ++s) i_byl[fill[lvl[s]]++] = s;
  }
  const char* pinned = nullptr;
  int rc = topo_image_get(img, &pinned);
  if (rc) return rc;
  SP_CUDA(cudaMemcpyAsync(ws + L.off_po, pinned, img.size(), cudaMemcpyHostToDevice, st));
  a.parent_offsets = reinterpret_cast<const int*>(ws + L.off_po);
  a.parent_ids = reinterpret_cast<const int*>(ws + L.off_pid);
  if (CAL) a.flux = reinterpret_cast<double*>(ws + L.off_flux);
  a.work_sc = reinterpret_cast<const int*>(ws + L.off_order);
  a.ticket = reinterpret_cast<int*>(ws + L.off_ticket);
  a.progress = reinterpret_cast<int*>(ws + L.off_progress);
  SP_CUDA(cudaMemsetAsync(ws + L.off_ticket, 0, L.off_flux - L.off_ticket, st));
  a.level_item_off = reinterpret_cast<const long long*>(ws + L.off_lvl_items);
  a.level_order_off = reinterpret_cast<const int*>(ws + L.off_lvl_order);
  a.n_levels = 2 * nl;
  stiff_group_kernel<<<1, 1024, 0, st>>>(S, nl, dims.n_members, reinterpret_cast<const int*>(ws + L.off_bylevel),
                                         reinterpret_cast<const int*>(ws + L.off_lvlstart), a.parent_offsets, a.parent_ids,
                                         a.sc_params, a.member_params, reinterpret_cast<double*>(ws + L.off_area),
                                         reinterpret_cast<int*>(ws + L.off_order), reinterpret_cast<int*>(ws + L.off_lvl_order),
                                         reinterpret_cast<long long*>(ws + L.off_lvl_items));
  // The padded item count depends on the split of each level, which only the device knows: the grid is sized for the
  // worst split (a level of n reaches x M members pads to at most ceil8(n M) + 8 items when cut in two); blocks and
  // warps beyond the actual count return at once.
  long long bound = 0;
  for (int l = 0; l < nl; ++l) {
    const long long n = (long long)(i_ls[l + 1] - i_ls[l]) * dims.n_members;
    bound += (n + 7) / 8 * 8 + ((dims.n_members % 8 != 0 && i_ls[l + 1] - i_ls[l] > 1) ? 8 : 0);
  }
  const LaunchConfig c = launch_config(
      {dims.n_members, dims.n_days, true, nl, (bound + qpb - 1) / qpb, opt.pilot_days, ws != nullptr, n_sm}, ov);
  if (c.n_epochs > 0) {
    a.epoch_days = c.epoch_days;
    a.n_epochs = c.n_epochs;
    a.epoch_done = reinterpret_cast<int*>(ws + L.off_epoch_done);
    a.carry = reinterpret_cast<QuadCarry*>(ws + L.off_carry);
    a.carry_stats = reinterpret_cast<double*>(ws + L.off_carry_stats);
    if (es != nullptr && es->flags_dev != nullptr && a.n_epochs <= es->capacity) {
      a.epoch_count = reinterpret_cast<unsigned*>(ws + L.off_epoch_count);
      a.epoch_flags_host = es->flags_dev;
      es->n_epochs = a.n_epochs;
      es->epoch_days = a.epoch_days;
    }
  }
  launch_quad<MODE, true>(c.minb, c.grid, smem, st, a);
  g_launches.fetch_add(2);
  SP_CUDA(cudaGetLastError());
  return SIMPLYP_OK;
}

KArgs base_args(const SimplypDims& dims, const SimplypOptions& opt, const double* forcing,
                const double* member_params, const double* sc_params) {
  KArgs a;
  memset(&a, 0, sizeof(a));
  a.M = dims.n_members; a.S = dims.n_sc; a.D = dims.n_days; a.Msc = dims.n_sc_param_sets;
  a.day_end = dims.n_days;
  a.V = dims.n_obs_series;
  a.topt = make_topt(opt);
  a.sc_qr0 = opt.sc_qr0;
  a.forcing = forcing; a.member_params = member_params; a.sc_params = sc_params;
  return a;
}

// Cached device buffers of the _host entry points: one cache (buffers + stream + lock) PER DEVICE, so that host
// threads driving different devices never touch each other's buffers; two threads on the same device take turns.
constexpr int MAX_DEVICES = 64;
struct HostCache {
  std::mutex lock;
  void* buf[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  size_t cap[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;     // device-to-host copies of finished epochs, beside the integration
  int* epoch_flags = nullptr;             // mapped pinned memory [EPOCH_FLAGS]: raised by the kernel, polled by the host
  int* epoch_flags_dev = nullptr;
};
constexpr int EPOCH_FLAGS = 4096;
HostCache g_cache[MAX_DEVICES];

int cache_get(HostCache& c, int slot, size_t bytes, void** out) {
  if (bytes == 0) bytes = 8;
  if (c.cap[slot] < bytes) {
    if (c.buf[slot]) cudaFree(c.buf[slot]);
    c.buf[slot] = nullptr;
    c.cap[slot] = 0;
    SP_CUDA(cudaMalloc(&c.buf[slot], bytes));
    c.cap[slot] = bytes;
  }
  *out = c.buf[slot];
  return SIMPLYP_OK;
}

// Makes `device` current for the calling thread and readies its cache; the caller holds c.lock.
int cache_select_device(int device, HostCache& c) {
  SP_CUDA(cudaSetDevice(device));
  if (!c.stream) SP_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
  if (!c.copy_stream) SP_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
  if (!c.epoch_flags) {
    SP_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&c.epoch_flags), sizeof(int) * EPOCH_FLAGS, cudaHostAllocMapped));
    SP_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&c.epoch_flags_dev), c.epoch_flags, 0));
  }
  return SIMPLYP_OK;
}

int check_device_index(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
  if (device < 0 || device >= n || device >= MAX_DEVICES) return fail(SIMPLYP_EINVAL, "device index out of range%s");
  return SIMPLYP_OK;
}

// ------------------------------------------------------------------------------------------ ensemble sampler
// One thread per walker of the active half (simplyp_mcmc.cuh holds the arithmetic).
__global__ void mcmc_propose_kernel(const SimplypMcmc mc, const SimplypMcmcState st, int half, double* member_params,
                                    double* sc_params) {
  const int H = mc.n_walkers / 2, K = mc.n_free, S = mc.n_sc;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= H) return;
  const long long t = *st.iteration;
  double* prop = st.proposals + (size_t)k * K;
  const int out = mcmc_propose_walker(mc, st.walkers, t, half, k, prop, st.log_z + k);
  st.out_of_box[k] = out;
  const int w = half * H + k;
  const double* src = out ? st.walkers + (size_t)w * K : prop;
  double* mrow = member_params + (size_t)w * SIMPLYP_NP_MEMBER;
  double* srow = sc_params + (mc.sc_per_member ? (size_t)w * S * SIMPLYP_NP_SC : 0);
  for (int i = 0; i < K; ++i) {
    const SimplypMcmcParam& p = mc.param[i];
    if (p.kind == SIMPLYP_MCMC_MEMBER) {
      mrow[p.index] = src[i];
    } else if (p.kind == SIMPLYP_MCMC_SC_AT) {
      srow[(size_t)p.pos * SIMPLYP_NP_SC + p.index] = src[i];
    } else {
      for (int s = 0; s < S; ++s) srow[(size_t)s * SIMPLYP_NP_SC + p.index] = src[i];
    }
  }
}

// Half 1 also stores the chain slot of the iteration: thread k writes walker k (half 0, final since the half-0
// accept) and walker H + k (its own).  The counter is advanced by mcmc_advance_kernel after every thread has read it.
__global__ void mcmc_accept_kernel(const SimplypMcmc mc, const SimplypMcmcState st, int half, const double* stats,
                                   const int64_t* diag) {
  const int H = mc.n_walkers / 2, K = mc.n_free, V = mc.n_obs_series, S = mc.n_sc;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= H) return;
  const long long t = *st.iteration;
  const double lp_new = st.out_of_box[k]
                            ? -INFINITY
                            : mcmc_member_lp(stats + (size_t)k * V * SIMPLYP_NSTAT, V, diag + (size_t)k * S * SIMPLYP_NDIAG, S);
  mcmc_accept_walker(mc, t, half, k, lp_new, st.log_z[k], st.proposals + (size_t)k * K, st.walkers, st.lp, st.accepted);
  if (half == 1 && (t + 1) % mc.thin == 0) {
    const long long slot = (t + 1) / mc.thin - 1 - st.chain_base;
    if (slot < 0 || slot >= st.n_saved) return;
    for (int w = k; w < 2 * H; w += H) {
      for (int i = 0; i < K; ++i)
        st.chain[((size_t)slot * mc.n_walkers + w) * K + i] = st.walkers[(size_t)w * K + i];
      st.chain_lp[(size_t)slot * mc.n_walkers + w] = st.lp[w];
    }
  }
}

__global__ void mcmc_advance_kernel(int64_t* iteration) { *iteration += 1; }

__global__ void mcmc_init_kernel(const SimplypMcmc mc, const SimplypMcmcState st, const double* stats,
                                 const int64_t* diag) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= mc.n_walkers) return;
  st.lp[w] = mcmc_member_lp(stats + (size_t)w * mc.n_obs_series * SIMPLYP_NSTAT, mc.n_obs_series,
                            diag + (size_t)w * mc.n_sc * SIMPLYP_NDIAG, mc.n_sc);
}

int check_mcmc(const SimplypMcmc* mc, const SimplypMcmcState* st) {
  if (!mc || !st) return fail(SIMPLYP_EINVAL, "mcmc: null argument%s");
  const int K = mc->n_free;
  if (K < 1 || K > SIMPLYP_MCMC_MAX_FREE) return fail(SIMPLYP_EINVAL, "mcmc: 1..SIMPLYP_MCMC_MAX_FREE free parameters%s");
  if (mc->n_walkers < 2 * K || mc->n_walkers % 2 != 0) return fail(SIMPLYP_EINVAL, "mcmc: an even number of walkers >= 2 K%s");
  if (mc->n_sc < 1 || mc->n_obs_series < 0 || mc->thin < 1) return fail(SIMPLYP_EINVAL, "mcmc: bad n_sc / n_obs_series / thin%s");
  if (!(mc->stretch > 1.0 && mc->stretch < INFINITY)) return fail(SIMPLYP_EINVAL, "mcmc: stretch scale must be > 1%s");
  for (int i = 0; i < K; ++i) {
    const SimplypMcmcParam& p = mc->param[i];
    if (!(p.lo < p.hi) || !std::isfinite(p.lo) || !std::isfinite(p.hi)) return fail(SIMPLYP_EINVAL, "mcmc: need finite lo < hi%s");
    if (p.kind == SIMPLYP_MCMC_MEMBER) {
      if (p.index < 0 || p.index >= SIMPLYP_NP_MEMBER) return fail(SIMPLYP_EINVAL, "mcmc: member column out of range%s");
    } else if (p.kind == SIMPLYP_MCMC_SC_ALL || p.kind == SIMPLYP_MCMC_SC_AT) {
      if (p.index < 0 || p.index >= SIMPLYP_NP_SC) return fail(SIMPLYP_EINVAL, "mcmc: SC row out of range%s");
      if (p.kind == SIMPLYP_MCMC_SC_AT && (p.pos < 0 || p.pos >= mc->n_sc)) return fail(SIMPLYP_EINVAL, "mcmc: SC position out of range%s");
      if (!mc->sc_per_member) return fail(SIMPLYP_EINVAL, "mcmc: SC targets need per-member sc_params%s");
    } else {
      return fail(SIMPLYP_EINVAL, "mcmc: unknown target kind%s");
    }
  }
  if (!st->walkers || !st->lp || !st->proposals || !st->log_z || !st->out_of_box || !st->iteration || !st->accepted)
    return fail(SIMPLYP_EINVAL, "mcmc: null state pointer%s");
  if (st->n_saved < 0 || (st->n_saved > 0 && (!st->chain || !st->chain_lp))) return fail(SIMPLYP_EINVAL, "mcmc: null chain%s");
  if (simplyp_device_count() <= 0) return fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
  return SIMPLYP_OK;
}

// ------------------------------------------------------------------------------------------ predictive bands
// Draws of V simulated series (sim_series_value, the values the fused statistics see) from the full output of a chunk
// of Mc members, optionally through the likelihood's error model (band_draw / band_epsilon): one block per
// (32 days, 32 members, series), 32 x 8 threads.  The out rows are read with the lane over days (consecutive rows of
// one member), the tile is transposed in shared memory and written with the lane over members, since
// draws[v][d][member_offset + m] is member-contiguous for the selection.  A member with a non-zero status word at any
// reach draws NaN everywhere (the sampler gives it -inf).
constexpr int DRAW_TILE = 32;
__global__ void __launch_bounds__(256) predictive_draws_kernel(const double* out, const double* member_params,
                                                               const double* sc_params, const int64_t* diag,
                                                               const int32_t* series_desc, int Mc, int S, int D,
                                                               int Msc, long long M_total, long long member_offset,
                                                               int obs_error, uint64_t seed, double* draws) {
  __shared__ double tile[DRAW_TILE][DRAW_TILE + 1];
  __shared__ int failed[DRAW_TILE];
  const int v = blockIdx.z, d0 = blockIdx.x * DRAW_TILE, m0 = blockIdx.y * DRAW_TILE;
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int s = series_desc[2 * v], kind = series_desc[2 * v + 1];
  if (ty == 0) {
    int f = 0;
    if (m0 + tx < Mc)
      for (int r = 0; r < S; ++r) f |= diag[((size_t)(m0 + tx) * S + r) * SIMPLYP_NDIAG + SIMPLYP_DG_STATUS] != 0;
    failed[tx] = f;
  }
  __syncthreads();
  const int d = d0 + tx;
  for (int j = ty; j < DRAW_TILE; j += blockDim.y) {
    const int m = m0 + j;
    if (m >= Mc || d >= D) continue;
    double y = NAN;
    if (!failed[j]) {
      const double* row = out + (((size_t)m * S + s) * D + d) * SIMPLYP_NOUT;
      const double* mp = member_params + (size_t)m * SIMPLYP_NP_MEMBER;
      const double A = sc_params[((size_t)(Msc > 1 ? m : 0) * S + s) * SIMPLYP_NP_SC + SIMPLYP_SC_A_CATCH];
      const double Qr = row[SIMPLYP_O_QR];
      y = sim_series_value(kind, Qr, row[SIMPLYP_O_MSUS_FLUX], row[SIMPLYP_O_TDP_FLUX], row[SIMPLYP_O_PP_FLUX], A,
                           sp_rcp(Qr), sp_rcp(A), mp[SIMPLYP_P_F_TDP]);
      if (obs_error)
        y = band_draw(y, mp[SIMPLYP_P_ERR_M0 + kind], band_epsilon(seed, (int)(member_offset + m), d, v));
    }
    tile[j][tx] = y;
  }
  __syncthreads();
  const int m = m0 + tx;
  for (int j = ty; j < DRAW_TILE; j += blockDim.y) {
    const int dd = d0 + j;
    if (m < Mc && dd < D) draws[((size_t)v * D + dd) * M_total + member_offset + m] = tile[tx][j];
  }
}

// np.nanquantile(x, q, axis=-1) of every row of x[R][N], with the mean and the count of the non-NaN entries.  The
// quantile values travel by value in the launch (a captured launch replays them).  Order statistics are exact: the
// entries are turned into order-preserving keys (nq_key, NaN last) and either sorted in shared memory
// (nanquantile_kernel, one block a row) or selected digit by digit in global memory (nq_*_kernel, longer rows).
struct NqArgs {
  int n_q;
  double q[SIMPLYP_NQ_MAX];
};
constexpr int NQ_THREADS = 1024;
constexpr int NQ_RANKS = 2 * SIMPLYP_NQ_MAX;     // two neighbours a quantile
constexpr int NQ_BINS = 256;                      // 8-bit digits, 8 passes
// Global-path workspace of one row: histograms [NQ_RANKS][NQ_BINS], then rank left / key prefix per neighbour, the
// weights g and the count.
struct NqRow {
  unsigned hist[NQ_RANKS][NQ_BINS];
  unsigned long long k[NQ_RANKS];
  unsigned long long prefix[NQ_RANKS];
  double g[SIMPLYP_NQ_MAX];
  long long n;
};

// Count and sum of the non-NaN entries of one row, reduced in a fixed order (the result does not depend on timing).
// Every thread returns the block's totals.
__device__ void nq_count_sum(const double* row, long long N, uint64_t* keys, long long* n_out, double* sum_out) {
  __shared__ double red_s[NQ_THREADS / 32];
  __shared__ long long red_n[NQ_THREADS / 32];
  double sum = 0.0;
  long long n = 0;
  for (long long i = threadIdx.x; i < N; i += blockDim.x) {
    const double v = row[i];
    if (keys) keys[i] = nq_key(v);
    if (v == v) { sum += v; ++n; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_down_sync(0xffffffffu, sum, o);
    n += __shfl_down_sync(0xffffffffu, n, o);
  }
  const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if ((threadIdx.x & 31) == 0) { red_s[w] = sum; red_n[w] = n; }
  __syncthreads();
  if (threadIdx.x < 32) {
    sum = threadIdx.x < nw ? red_s[threadIdx.x] : 0.0;
    n = threadIdx.x < nw ? red_n[threadIdx.x] : 0;
    for (int o = 16; o > 0; o >>= 1) {
      sum += __shfl_down_sync(0xffffffffu, sum, o);
      n += __shfl_down_sync(0xffffffffu, n, o);
    }
    if (threadIdx.x == 0) { red_s[0] = sum; red_n[0] = n; }
  }
  __syncthreads();
  *sum_out = red_s[0];
  *n_out = red_n[0];
}

// Rows of N <= the shared-memory capacity: keys[N] in dynamic shared memory, sorted by a bitonic network on the next
// power of two.  The comparators all put the smaller key first (the first step of every merge compares mirrored
// positions), so the virtual padding of largest keys never moves and every comparator that reaches it is skipped.
__global__ void __launch_bounds__(NQ_THREADS) nanquantile_kernel(const double* x, long long R, long long N,
                                                                 const NqArgs qa, double* quant, double* mean,
                                                                 int64_t* count) {
  extern __shared__ uint64_t keys[];
  const long long r = blockIdx.x;
  long long n;
  double sum;
  nq_count_sum(x + r * N, N, keys, &n, &sum);
  long long P = 1;
  while (P < N) P <<= 1;
  for (long long k = 2; k <= P; k <<= 1) {
    for (long long j = k >> 1; j > 0; j >>= 1) {
      for (long long t = threadIdx.x; t < P / 2; t += blockDim.x) {
        const long long i = 2 * j * (t / j) + (t % j);
        const long long p = (j == (k >> 1)) ? (i ^ (k - 1)) : (i + j);
        if (p < N) {
          const uint64_t a = keys[i], b = keys[p];
          if (b < a) { keys[i] = b; keys[p] = a; }
        }
      }
      __syncthreads();
    }
  }
  if (threadIdx.x < qa.n_q) {
    double res = NAN;
    if (n > 0) {
      long long lo, hi;
      double g;
      nq_index(n, qa.q[threadIdx.x], &lo, &hi, &g);
      res = nq_lerp(nq_value(keys[lo]), nq_value(keys[hi]), g);
    }
    quant[(size_t)threadIdx.x * R + r] = res;
  }
  if (threadIdx.x == 0) {
    mean[r] = n > 0 ? sum / (double)n : NAN;
    count[r] = n;
  }
}

// Longer rows, 1: count, mean and the ranks of the neighbours of every quantile; histograms zeroed.
__global__ void __launch_bounds__(NQ_THREADS) nq_prepare_kernel(const double* x, long long N, const NqArgs qa,
                                                                NqRow* ws, double* mean, int64_t* count) {
  const long long r = blockIdx.x;
  NqRow& w = ws[r];
  long long n;
  double sum;
  nq_count_sum(x + r * N, N, nullptr, &n, &sum);
  for (int i = threadIdx.x; i < NQ_RANKS * NQ_BINS; i += blockDim.x) (&w.hist[0][0])[i] = 0u;
  if (threadIdx.x < qa.n_q && n > 0) {
    long long lo, hi;
    double g;
    nq_index(n, qa.q[threadIdx.x], &lo, &hi, &g);
    w.k[2 * threadIdx.x] = (unsigned long long)lo;
    w.k[2 * threadIdx.x + 1] = (unsigned long long)hi;
    w.prefix[2 * threadIdx.x] = w.prefix[2 * threadIdx.x + 1] = 0ull;
    w.g[threadIdx.x] = g;
  }
  if (threadIdx.x == 0) {
    w.n = n;
    mean[r] = n > 0 ? sum / (double)n : NAN;
    count[r] = n;
  }
}

// 2: the histogram of digit `pass` (from the top) of the keys that share each neighbour's prefix so far; blocks of
// 256 threads over a slice (blockIdx.y) of one row (blockIdx.x), counted in shared memory first.
constexpr int NQ_HIST_THREADS = 256, NQ_HIST_PER_THREAD = 16;
__global__ void __launch_bounds__(NQ_HIST_THREADS) nq_hist_kernel(const double* x, long long N, int n_q, int pass,
                                                                  NqRow* ws) {
  __shared__ unsigned h[NQ_RANKS][NQ_BINS];
  __shared__ unsigned long long pre[NQ_RANKS];
  const long long r = blockIdx.x;
  NqRow& w = ws[r];
  const int nr = 2 * n_q;
  for (int i = threadIdx.x; i < NQ_RANKS * NQ_BINS; i += blockDim.x) (&h[0][0])[i] = 0u;
  if (threadIdx.x < nr) pre[threadIdx.x] = w.prefix[threadIdx.x];
  __syncthreads();
  if (w.n == 0) return;
  const int shift = 56 - 8 * pass;
  const unsigned long long mask = pass == 0 ? 0ull : (~0ull << (shift + 8));
  const long long base = (long long)blockIdx.y * NQ_HIST_THREADS * NQ_HIST_PER_THREAD;
  const double* row = x + r * N;
  for (int e = 0; e < NQ_HIST_PER_THREAD; ++e) {
    const long long i = base + (long long)e * NQ_HIST_THREADS + threadIdx.x;
    if (i >= N) break;
    const uint64_t key = nq_key(row[i]);
    const unsigned digit = (unsigned)(key >> shift) & 0xFFu;
    for (int j = 0; j < nr; ++j)
      if (((key ^ pre[j]) & mask) == 0) atomicAdd(&h[j][digit], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nr * NQ_BINS; i += blockDim.x) {
    const unsigned c = (&h[0][0])[i];
    if (c) atomicAdd(&(&w.hist[0][0])[i], c);
  }
}

// 3: every neighbour takes the digit whose cumulative count passes its rank; the histograms are zeroed for the next
// pass.  After the last pass the prefixes are the keys of the neighbours and the quantiles are interpolated.
__global__ void nq_pick_kernel(long long R, const NqArgs qa, int pass, NqRow* ws, double* quant) {
  const long long r = blockIdx.x;
  NqRow& w = ws[r];
  const int j = threadIdx.x, nr = 2 * qa.n_q;
  if (j < nr && w.n > 0) {
    const int shift = 56 - 8 * pass;
    unsigned long long k = w.k[j], below = 0;
    int b = 0;
    for (; b < NQ_BINS - 1; ++b) {
      const unsigned long long c = w.hist[j][b];
      if (below + c > k) break;
      below += c;
    }
    w.k[j] = k - below;
    w.prefix[j] |= (unsigned long long)b << shift;
    for (int i = 0; i < NQ_BINS; ++i) w.hist[j][i] = 0u;
  }
  if (pass == 7) {
    __syncthreads();
    if (j < qa.n_q)
      quant[(size_t)j * R + r] =
          w.n > 0 ? nq_lerp(nq_value(w.prefix[2 * j]), nq_value(w.prefix[2 * j + 1]), w.g[j]) : NAN;
  }
}

// Rows up to this many entries take the shared-memory path on the current device.
long long nq_shared_cap() {
  int dev = 0, optin = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
    return 0;
  return (optin - 1024) / (long long)sizeof(uint64_t);   // (1 KB for the reductions' static shared memory)
}

}  // namespace

// ============================================================================================ C-ABI
extern "C" {

int simplyp_abi_version(void) { return SIMPLYP_ABI_VERSION; }
const char* simplyp_version(void) { return "simplyp_b200 0.1.0 (sm_100a)"; }
const char* simplyp_last_error(void) { return g_err; }

int simplyp_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

void simplyp_default_options(SimplypOptions* opt) {
  if (!opt) return;
  memset(opt, 0, sizeof(*opt));
  opt->rtol = 1e-7;
  opt->atol = 1e-10;
  opt->step_len = 1.0;
  opt->max_steps_per_day = 5000;
  opt->run_mode_cal = 1;
  opt->strict_quirks = 1;
}

int simplyp_topology_levels(int32_t n_sc, const int32_t* parent_offsets, const int32_t* parent_ids,
                            int32_t* levels) {
  if (n_sc < 0 || !parent_offsets || (!parent_ids && parent_offsets[n_sc] > 0) || !levels)
    return fail(SIMPLYP_EINVAL, "null argument%s");
  std::vector<int> lvl;
  const int nl = topology_levels(n_sc, parent_offsets, parent_ids, lvl);
  if (nl < 0) return fail(SIMPLYP_EINVAL, "topology: parents must precede children in run order%s");
  for (int s = 0; s < n_sc; ++s) levels[s] = lvl[s];
  return nl;
}

int64_t simplyp_workspace_bytes(const SimplypDims* dims, int calibrate) {
  if (!dims) return SIMPLYP_EINVAL;
  return (int64_t)ws_layout(*dims, dims->reserved[0], (calibrate & 1) != 0, (calibrate & 2) != 0).total;
}

static int run_device_impl(const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                           const double* member_params, const double* sc_params, const int32_t* parent_offsets,
                           const int32_t* parent_ids, double* out, int64_t* diag, void* workspace, void* stream,
                           EpochStream* es) {
  int rc = check_common(dims, opt, forcing, member_params, sc_params, parent_offsets);
  if (rc) return rc;
  if (!out) return fail(SIMPLYP_EINVAL, "null output%s");
  if (simplyp_device_count() <= 0) return fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
  if (dims->n_days == 0) return SIMPLYP_OK;
  KArgs a = base_args(*dims, *opt, forcing, member_params, sc_params);
  a.out = out;
  a.diag = reinterpret_cast<long long*>(diag);
  return launch_levels<false>(*dims, *opt, a, parent_offsets, parent_ids, static_cast<char*>(workspace),
                              static_cast<cudaStream_t>(stream), es);
}

int simplyp_run_device(const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                       const double* member_params, const double* sc_params, const int32_t* parent_offsets,
                       const int32_t* parent_ids, double* out, int64_t* diag, void* workspace, void* stream) {
  return run_device_impl(dims, opt, forcing, member_params, sc_params, parent_offsets, parent_ids, out, diag, workspace,
                         stream, nullptr);
}

static int calibrate_device_impl(const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                                 const double* member_params, const double* sc_params,
                                 const int32_t* parent_offsets, const int32_t* parent_ids, const double* obs,
                                 const int32_t* obs_desc, double* stats, int64_t* diag, void* workspace,
                                 void* stream, const SimplypPeerGather* pg) {
  int rc = check_common(dims, opt, forcing, member_params, sc_params, parent_offsets);
  if (rc) return rc;
  if (dims->n_obs_series < 0 || (dims->n_obs_series > 0 && (!obs || !obs_desc || !stats)))
    return fail(SIMPLYP_EINVAL, "null observation/statistics argument%s");
  if (!workspace) return fail(SIMPLYP_EINVAL, "workspace required%s");
  if (simplyp_device_count() <= 0) return fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int V = dims->n_obs_series;
  const bool ranks = opt->rank_stats != 0 && V > 0 && dims->n_days > 0;
  const WsLayout L = ws_layout(*dims, parent_offsets[dims->n_sc], true, ranks);
  char* ws = static_cast<char*>(workspace);
  KArgs a = base_args(*dims, *opt, forcing, member_params, sc_params);
  a.diag = reinterpret_cast<long long*>(diag);
  a.obs = obs;
  a.obs_desc = obs_desc;
  a.stats = stats;
  if (pg != nullptr) {
    a.n_peers = pg->n_ranks;
    a.my_rank = pg->rank;
    a.member_offset = pg->member_offset;
    for (int r = 0; r < pg->n_ranks; ++r) a.peer_stats[r] = pg->stats_bufs[r];
  }
  a.obs_const = reinterpret_cast<const double*>(ws + L.off_oc);
  double* obs_rank = reinterpret_cast<double*>(ws + L.off_obs_rank);
  if (V > 0) {
    SP_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * SIMPLYP_NSTAT * (size_t)dims->n_members * V, st));
    if (dims->n_days > 0) {
      obs_const_kernel<<<V, 256, 0, st>>>(obs, dims->n_days, reinterpret_cast<double*>(ws + L.off_oc),
                                          reinterpret_cast<double*>(ws + L.off_obs_log));
      a.obs_log = reinterpret_cast<const double*>(ws + L.off_obs_log);
      g_launches.fetch_add(1);
      if (ranks) {
        obs_rank_kernel<<<V, 256, 0, st>>>(obs, dims->n_days, obs_rank, reinterpret_cast<double*>(ws + L.off_oc));
        g_launches.fetch_add(1);
        a.sim_obs = reinterpret_cast<double*>(ws + L.off_sim_obs);
        // a day without a finite simulated value must read as NaN (dropped pair)
        SP_CUDA(cudaMemsetAsync(a.sim_obs, 0xff, sizeof(double) * (size_t)dims->n_members * V * dims->n_days, st));
      }
      SP_CUDA(cudaGetLastError());
    }
  }
  if (dims->n_days == 0) return SIMPLYP_OK;
  rc = launch_levels<true>(*dims, *opt, a, parent_offsets, parent_ids, ws, st);
  if (rc) return rc;
  if (ranks) {
    // shared memory: sim values + obs ranks of one series, at most one entry per day; longer records take the
    // global-memory variant
    const int cap_max = (200 * 1024) / 16;
    if (dims->n_days <= cap_max) {
      const int cap = dims->n_days;
      const size_t smem = (size_t)cap * 2 * sizeof(double);
      if (smem > 48 * 1024)
        SP_CUDA(cudaFuncSetAttribute(spearman_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      spearman_kernel<<<(unsigned)((size_t)dims->n_members * V), 128, smem, st>>>(
          a.sim_obs, obs_rank, a.obs_const, V, dims->n_days, cap, stats);
    } else {
      spearman_long_kernel<<<(unsigned)((size_t)dims->n_members * V), 128, 0, st>>>(
          a.sim_obs, obs_rank, a.obs_const, V, dims->n_days, stats);
    }
    g_launches.fetch_add(1);
    SP_CUDA(cudaGetLastError());
  }
  if (pg != nullptr && pg->n_ranks > 1) {
    PeerFlags f;
    for (int r = 0; r < SIMPLYP_MAX_RANKS; ++r) f.bufs[r] = r < pg->n_ranks ? pg->flag_bufs[r] : nullptr;
    long long* status_word = diag ? reinterpret_cast<long long*>(diag) + SIMPLYP_DG_STATUS : nullptr;
    peer_flag_kernel<<<1, 32, 0, st>>>(f, pg->n_ranks, pg->rank, (int)pg->step, status_word);
    g_launches.fetch_add(1);
    SP_CUDA(cudaGetLastError());
  }
  return SIMPLYP_OK;
}

int simplyp_calibrate_device(const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                             const double* member_params, const double* sc_params,
                             const int32_t* parent_offsets, const int32_t* parent_ids, const double* obs,
                             const int32_t* obs_desc, double* stats, int64_t* diag, void* workspace,
                             void* stream) {
  return calibrate_device_impl(dims, opt, forcing, member_params, sc_params, parent_offsets, parent_ids, obs, obs_desc,
                               stats, diag, workspace, stream, nullptr);
}

int simplyp_calibrate_gather_device(const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                                    const double* member_params, const double* sc_params,
                                    const int32_t* parent_offsets, const int32_t* parent_ids, const double* obs,
                                    const int32_t* obs_desc, const SimplypPeerGather* gather, int64_t* diag,
                                    void* workspace, void* stream) {
  if (!gather || !dims) return fail(SIMPLYP_EINVAL, "null gather descriptor%s");
  if (gather->n_ranks < 1 || gather->n_ranks > SIMPLYP_MAX_RANKS || gather->rank < 0 || gather->rank >= gather->n_ranks)
    return fail(SIMPLYP_EINVAL, "gather: 1..SIMPLYP_MAX_RANKS ranks, rank inside%s");
  if (gather->member_offset < 0 || gather->member_offset + dims->n_members > gather->n_members_total)
    return fail(SIMPLYP_EINVAL, "gather: this rank's members must lie inside the ensemble%s");
  if (opt && opt->rank_stats) return fail(SIMPLYP_EINVAL, "gather: rank statistics are filled by a later kernel, use the plain entry point%s");
  for (int r = 0; r < gather->n_ranks; ++r)
    if (!gather->stats_bufs[r] || !gather->flag_bufs[r]) return fail(SIMPLYP_EINVAL, "gather: null peer buffer%s");
  double* stats = gather->stats_bufs[gather->rank] +
                  (size_t)gather->member_offset * (dims->n_obs_series > 0 ? dims->n_obs_series : 0) * SIMPLYP_NSTAT;
  return calibrate_device_impl(dims, opt, forcing, member_params, sc_params, parent_offsets, parent_ids, obs, obs_desc,
                               stats, diag, workspace, stream, gather);
}

int simplyp_peer_alloc(int64_t bytes, void** dptr) {
  if (!dptr || bytes <= 0) return fail(SIMPLYP_EINVAL, "peer_alloc: bad argument%s");
  if (simplyp_device_count() <= 0) return fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
  SP_CUDA(cudaMalloc(dptr, (size_t)bytes));
  SP_CUDA(cudaMemset(*dptr, 0, (size_t)bytes));
  SP_CUDA(cudaDeviceSynchronize());
  return SIMPLYP_OK;
}
int simplyp_peer_free(void* dptr) {
  if (dptr) SP_CUDA(cudaFree(dptr));
  return SIMPLYP_OK;
}
int simplyp_ipc_export(const void* dptr, unsigned char handle[64]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  if (!dptr || !handle) return fail(SIMPLYP_EINVAL, "ipc_export: null argument%s");
  cudaIpcMemHandle_t h;
  SP_CUDA(cudaIpcGetMemHandle(&h, const_cast<void*>(dptr)));
  memcpy(handle, &h, 64);
  return SIMPLYP_OK;
}
int simplyp_ipc_import(const unsigned char handle[64], void** dptr) {
  if (!dptr || !handle) return fail(SIMPLYP_EINVAL, "ipc_import: null argument%s");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  SP_CUDA(cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
  return SIMPLYP_OK;
}
int simplyp_ipc_close(void* dptr) {
  if (dptr) SP_CUDA(cudaIpcCloseMemHandle(dptr));
  return SIMPLYP_OK;
}

int simplyp_run_host(int device, const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                     const double* member_params, const double* sc_params, const int32_t* parent_offsets,
                     const int32_t* parent_ids, double* out, int64_t* diag) {
  int rc = check_common(dims, opt, forcing, member_params, sc_params, parent_offsets);
  if (rc) return rc;
  if (!out) return fail(SIMPLYP_EINVAL, "null output%s");
  rc = check_device_index(device);
  if (rc) return rc;
  HostCache& hc = g_cache[device];
  std::lock_guard<std::mutex> guard(hc.lock);
  rc = cache_select_device(device, hc);
  if (rc) return rc;
  cudaStream_t st = hc.stream;
  const size_t M = dims->n_members, S = dims->n_sc, D = dims->n_days, Msc = dims->n_sc_param_sets;
  const size_t b_forc = sizeof(double) * SIMPLYP_NF * D, b_mp = sizeof(double) * SIMPLYP_NP_MEMBER * M;
  const size_t b_sc = sizeof(double) * SIMPLYP_NP_SC * Msc * S, b_out = sizeof(double) * SIMPLYP_NOUT * M * S * D;
  const size_t b_diag = sizeof(int64_t) * SIMPLYP_NDIAG * M * S;
  SimplypDims d2 = *dims;
  d2.reserved[0] = parent_offsets[S];
  const size_t b_ws = (size_t)simplyp_workspace_bytes(&d2, 0);
  void *d_forc, *d_mp, *d_sc, *d_out, *d_diag, *d_ws;
  if ((rc = cache_get(hc, 0, b_forc, &d_forc)) || (rc = cache_get(hc, 1, b_mp, &d_mp)) || (rc = cache_get(hc, 2, b_sc, &d_sc)) ||
      (rc = cache_get(hc, 3, b_out, &d_out)) || (rc = cache_get(hc, 4, b_diag, &d_diag)) || (rc = cache_get(hc, 5, b_ws, &d_ws)))
    return rc;
  SP_CUDA(cudaMemcpyAsync(d_forc, forcing, b_forc, cudaMemcpyHostToDevice, st));
  SP_CUDA(cudaMemcpyAsync(d_mp, member_params, b_mp, cudaMemcpyHostToDevice, st));
  SP_CUDA(cudaMemcpyAsync(d_sc, sc_params, b_sc, cudaMemcpyHostToDevice, st));
  EpochStream es;
  es.flags_dev = hc.epoch_flags_dev;
  es.capacity = EPOCH_FLAGS;
  memset(hc.epoch_flags, 0, sizeof(int) * EPOCH_FLAGS);       // (the previous call on this device has finished: see the lock)
  rc = run_device_impl(dims, opt, (const double*)d_forc, (const double*)d_mp, (const double*)d_sc, parent_offsets,
                       parent_ids, (double*)d_out, (int64_t*)d_diag, d_ws, st, &es);
  if (rc) return rc;
  if (es.n_epochs > 1) {
    // A network swept in epochs: the rows of epoch e (days [e E, (e+1) E) of every item: a strided 2-D block of the
    // [M][S][D][25] array) are final once every item has finished it, and leave on the copy stream while the later
    // epochs integrate.  The kernel raises one mapped flag per epoch; the last epoch is copied after the kernel.
    const size_t row = sizeof(double) * SIMPLYP_NOUT, pitch = row * D;
    int copied = 0;
    volatile int* flags = hc.epoch_flags;
    while (copied + 1 < es.n_epochs) {
      if (!flags[copied]) {
        if (cudaStreamQuery(st) != cudaErrorNotReady) break;   // finished (or failed): the rest is copied below
        std::this_thread::sleep_for(std::chrono::microseconds(20));
        continue;
      }
      const size_t d0 = (size_t)copied * es.epoch_days;
      SP_CUDA(cudaMemcpy2DAsync(reinterpret_cast<char*>(out) + row * d0, pitch, reinterpret_cast<const char*>(d_out) + row * d0,
                                pitch, row * es.epoch_days, M * S, cudaMemcpyDeviceToHost, hc.copy_stream));
      ++copied;
    }
    SP_CUDA(cudaStreamSynchronize(st));
    const size_t d0 = (size_t)copied * es.epoch_days;
    SP_CUDA(cudaMemcpy2DAsync(reinterpret_cast<char*>(out) + row * d0, pitch, reinterpret_cast<const char*>(d_out) + row * d0,
                              pitch, row * (D - d0), M * S, cudaMemcpyDeviceToHost, hc.copy_stream));
    if (diag) SP_CUDA(cudaMemcpyAsync(diag, d_diag, b_diag, cudaMemcpyDeviceToHost, hc.copy_stream));
    SP_CUDA(cudaStreamSynchronize(hc.copy_stream));
    return SIMPLYP_OK;
  }
  SP_CUDA(cudaMemcpyAsync(out, d_out, b_out, cudaMemcpyDeviceToHost, st));
  if (diag) SP_CUDA(cudaMemcpyAsync(diag, d_diag, b_diag, cudaMemcpyDeviceToHost, st));
  SP_CUDA(cudaStreamSynchronize(st));
  return SIMPLYP_OK;
}

int simplyp_calibrate_host(int device, const SimplypDims* dims, const SimplypOptions* opt, const double* forcing,
                           const double* member_params, const double* sc_params, const int32_t* parent_offsets,
                           const int32_t* parent_ids, const double* obs, const int32_t* obs_desc, double* stats,
                           int64_t* diag) {
  int rc = check_common(dims, opt, forcing, member_params, sc_params, parent_offsets);
  if (rc) return rc;
  if (dims->n_obs_series <= 0 || !obs || !obs_desc || !stats)
    return fail(SIMPLYP_EINVAL, "observations and statistics buffers required%s");
  // the rows are in host memory here, so they are checked before any device work (the device entry points take them
  // as a precondition: a reach outside 0..S-1 is never finalised, a kind outside 0..5 reads another parameter)
  for (int v = 0; v < dims->n_obs_series; ++v) {
    const int32_t sc = obs_desc[2 * v], kind = obs_desc[2 * v + 1];
    if (sc < 0 || sc >= dims->n_sc || kind < 0 || kind >= SIMPLYP_NVARKIND) {
      char row[160];
      snprintf(row, sizeof(row), "obs_desc row %d = (%d, %d): reach must be in 0..%d and kind in 0..%d", v, (int)sc,
               (int)kind, dims->n_sc - 1, SIMPLYP_NVARKIND - 1);
      return fail(SIMPLYP_EINVAL, "%s", row);
    }
  }
  rc = check_device_index(device);
  if (rc) return rc;
  HostCache& hc = g_cache[device];
  std::lock_guard<std::mutex> guard(hc.lock);
  rc = cache_select_device(device, hc);
  if (rc) return rc;
  cudaStream_t st = hc.stream;
  const size_t M = dims->n_members, S = dims->n_sc, D = dims->n_days, Msc = dims->n_sc_param_sets;
  const size_t V = dims->n_obs_series;
  const size_t b_forc = sizeof(double) * SIMPLYP_NF * D, b_mp = sizeof(double) * SIMPLYP_NP_MEMBER * M;
  const size_t b_sc = sizeof(double) * SIMPLYP_NP_SC * Msc * S;
  const size_t b_obs = sizeof(double) * V * D, b_desc = sizeof(int32_t) * 2 * V;
  const size_t b_stats = sizeof(double) * SIMPLYP_NSTAT * M * V, b_diag = sizeof(int64_t) * SIMPLYP_NDIAG * M * S;
  SimplypDims d2 = *dims;
  d2.reserved[0] = parent_offsets[S];
  const size_t b_ws = (size_t)simplyp_workspace_bytes(&d2, opt->rank_stats ? 3 : 1);
  void *d_forc, *d_mp, *d_sc, *d_obs, *d_desc, *d_stats, *d_diag, *d_ws;
  if ((rc = cache_get(hc, 0, b_forc, &d_forc)) || (rc = cache_get(hc, 1, b_mp, &d_mp)) || (rc = cache_get(hc, 2, b_sc, &d_sc)) ||
      (rc = cache_get(hc, 3, b_stats, &d_stats)) || (rc = cache_get(hc, 4, b_diag, &d_diag)) ||
      (rc = cache_get(hc, 5, b_ws, &d_ws)) || (rc = cache_get(hc, 6, b_obs, &d_obs)) || (rc = cache_get(hc, 7, b_desc, &d_desc)))
    return rc;
  SP_CUDA(cudaMemcpyAsync(d_forc, forcing, b_forc, cudaMemcpyHostToDevice, st));
  SP_CUDA(cudaMemcpyAsync(d_mp, member_params, b_mp, cudaMemcpyHostToDevice, st));
  SP_CUDA(cudaMemcpyAsync(d_sc, sc_params, b_sc, cudaMemcpyHostToDevice, st));
  SP_CUDA(cudaMemcpyAsync(d_obs, obs, b_obs, cudaMemcpyHostToDevice, st));
  SP_CUDA(cudaMemcpyAsync(d_desc, obs_desc, b_desc, cudaMemcpyHostToDevice, st));
  rc = simplyp_calibrate_device(dims, opt, (const double*)d_forc, (const double*)d_mp, (const double*)d_sc,
                                parent_offsets, parent_ids, (const double*)d_obs, (const int32_t*)d_desc,
                                (double*)d_stats, (int64_t*)d_diag, d_ws, st);
  if (rc) return rc;
  SP_CUDA(cudaMemcpyAsync(stats, d_stats, b_stats, cudaMemcpyDeviceToHost, st));
  if (diag) SP_CUDA(cudaMemcpyAsync(diag, d_diag, b_diag, cudaMemcpyDeviceToHost, st));
  SP_CUDA(cudaStreamSynchronize(st));
  return SIMPLYP_OK;
}

int simplyp_sum_to_waterbody_device(const SimplypDims* dims, const double* out, const double* sc_params,
                                    const double* member_params, const int32_t* reaches, int32_t n_reaches,
                                    double* waterbody, void* stream) {
  if (!dims || !out || !sc_params || !member_params || !reaches || !waterbody)
    return fail(SIMPLYP_EINVAL, "null argument%s");
  if (n_reaches <= 0 || n_reaches > dims->n_sc) return fail(SIMPLYP_EINVAL, "bad number of waterbody reaches%s");
  if (simplyp_device_count() <= 0) return fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
  const long long n = (long long)dims->n_members * dims->n_days;
  if (n == 0) return SIMPLYP_OK;
  waterbody_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      out, sc_params, member_params, reaches, n_reaches, dims->n_members, dims->n_sc, dims->n_days,
      dims->n_sc_param_sets, waterbody);
  g_launches.fetch_add(1);
  SP_CUDA(cudaGetLastError());
  return SIMPLYP_OK;
}

int simplyp_thornthwaite_pet_device(int32_t n_days, int32_t n_months, const double* t_air, int32_t t_stride,
                                    const int32_t* month_start, const int32_t* year_is_leap, double latitude_deg,
                                    double* pet, int32_t pet_stride, void* stream) {
  if (!t_air || !month_start || !year_is_leap || !pet) return fail(SIMPLYP_EINVAL, "null argument%s");
  if (n_days <= 0 || n_months <= 0 || n_months % 12 != 0 || t_stride <= 0 || pet_stride <= 0)
    return fail(SIMPLYP_EINVAL, "PET needs whole calendar years (n_months a multiple of 12)%s");
  if (n_months > 2880) return fail(SIMPLYP_EINVAL, "PET: more than 240 years%s");
  if (!(latitude_deg >= -90.0 && latitude_deg <= 90.0)) return fail(SIMPLYP_EINVAL, "latitude outside -90..90 degrees%s");
  if (simplyp_device_count() <= 0) return fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
  thornthwaite_kernel<<<1, 256, sizeof(double) * 2 * (size_t)n_months, static_cast<cudaStream_t>(stream)>>>(
      n_days, n_months, t_air, t_stride, month_start, year_is_leap, latitude_deg * (M_PI / 180.0), pet, pet_stride);
  g_launches.fetch_add(1);
  SP_CUDA(cudaGetLastError());
  return SIMPLYP_OK;
}

int simplyp_mcmc_propose_device(const SimplypMcmc* mc, const SimplypMcmcState* state, int half,
                                double* member_params, double* sc_params, void* stream) {
  int rc = check_mcmc(mc, state);
  if (rc) return rc;
  if (half != 0 && half != 1) return fail(SIMPLYP_EINVAL, "mcmc: half must be 0 or 1%s");
  if (!member_params || !sc_params) return fail(SIMPLYP_EINVAL, "mcmc: null parameter rows%s");
  const int H = mc->n_walkers / 2;
  mcmc_propose_kernel<<<(H + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(*mc, *state, half,
                                                                                       member_params, sc_params);
  g_launches.fetch_add(1);
  SP_CUDA(cudaGetLastError());
  return SIMPLYP_OK;
}

int simplyp_mcmc_accept_device(const SimplypMcmc* mc, const SimplypMcmcState* state, int half,
                               const double* stats, const int64_t* diag, void* stream) {
  int rc = check_mcmc(mc, state);
  if (rc) return rc;
  if (half != 0 && half != 1) return fail(SIMPLYP_EINVAL, "mcmc: half must be 0 or 1%s");
  if (!diag || (mc->n_obs_series > 0 && !stats)) return fail(SIMPLYP_EINVAL, "mcmc: null statistics%s");
  const int H = mc->n_walkers / 2;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  mcmc_accept_kernel<<<(H + 127) / 128, 128, 0, st>>>(*mc, *state, half, stats, diag);
  g_launches.fetch_add(1);
  SP_CUDA(cudaGetLastError());
  if (half == 1) {
    mcmc_advance_kernel<<<1, 1, 0, st>>>(state->iteration);
    g_launches.fetch_add(1);
    SP_CUDA(cudaGetLastError());
  }
  return SIMPLYP_OK;
}

int simplyp_mcmc_init_device(const SimplypMcmc* mc, const SimplypMcmcState* state, const double* stats,
                             const int64_t* diag, void* stream) {
  int rc = check_mcmc(mc, state);
  if (rc) return rc;
  if (!diag || (mc->n_obs_series > 0 && !stats)) return fail(SIMPLYP_EINVAL, "mcmc: null statistics%s");
  mcmc_init_kernel<<<(mc->n_walkers + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(*mc, *state, stats,
                                                                                               diag);
  g_launches.fetch_add(1);
  SP_CUDA(cudaGetLastError());
  return SIMPLYP_OK;
}

int simplyp_predictive_draws_device(const SimplypDims* dims, const double* out, const double* member_params,
                                    const double* sc_params, const int64_t* diag, const int32_t* series_desc,
                                    int32_t n_series, double* draws, int64_t n_members_total, int64_t member_offset,
                                    int32_t obs_error, uint64_t seed, void* stream) {
  if (!dims || !out || !member_params || !sc_params || !diag || !series_desc || !draws)
    return fail(SIMPLYP_EINVAL, "predictive draws: null argument%s");
  const int M = dims->n_members, S = dims->n_sc, D = dims->n_days, Msc = dims->n_sc_param_sets;
  if (M < 1 || M > 65535 * DRAW_TILE || S < 1 || D < 0 || (Msc != 1 && Msc != M) || n_series < 1 || n_series > 65535)
    return fail(SIMPLYP_EINVAL, "predictive draws: bad dims (1 <= M <= 2097120 a chunk, S >= 1, D >= 0, Msc = 1 or M, "
                                "1..65535 series)%s");
  if (member_offset < 0 || n_members_total > INT32_MAX || member_offset + M > n_members_total)
    return fail(SIMPLYP_EINVAL, "predictive draws: members outside 0..n_members_total - 1 (at most 2^31 - 1)%s");
  if (obs_error != 0 && obs_error != 1) return fail(SIMPLYP_EINVAL, "predictive draws: obs_error must be 0 or 1%s");
  if (simplyp_device_count() <= 0) return fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
  if (D == 0) return SIMPLYP_OK;
  const dim3 grid((unsigned)((D + DRAW_TILE - 1) / DRAW_TILE), (unsigned)((M + DRAW_TILE - 1) / DRAW_TILE),
                  (unsigned)n_series);
  predictive_draws_kernel<<<grid, dim3(DRAW_TILE, 8), 0, static_cast<cudaStream_t>(stream)>>>(
      out, member_params, sc_params, diag, series_desc, M, S, D, Msc, n_members_total, member_offset, obs_error, seed,
      draws);
  g_launches.fetch_add(1);
  SP_CUDA(cudaGetLastError());
  return SIMPLYP_OK;
}

int64_t simplyp_nanquantile_workspace_bytes(int64_t n_rows, int64_t n_cols) {
  if (n_rows < 0 || n_cols < 0) return fail(SIMPLYP_EINVAL, "nanquantile: negative dims%s");
  if (n_cols <= nq_shared_cap()) return 0;
  return n_rows * (int64_t)sizeof(NqRow);
}

int simplyp_nanquantile_device(const double* x, int64_t n_rows, int64_t n_cols, const double* q, int32_t n_q,
                               double* quantiles, double* mean, int64_t* count, void* workspace,
                               int64_t workspace_bytes, void* stream) {
  if (!x || !q || !quantiles || !mean || !count) return fail(SIMPLYP_EINVAL, "nanquantile: null argument%s");
  if (n_rows < 0 || n_rows > INT32_MAX || n_cols < 1 || n_q < 1 || n_q > SIMPLYP_NQ_MAX)
    return fail(SIMPLYP_EINVAL, "nanquantile: bad dims (0..2^31 - 1 rows, n_cols >= 1, 1..SIMPLYP_NQ_MAX quantiles)%s");
  NqArgs qa;
  qa.n_q = n_q;
  for (int i = 0; i < SIMPLYP_NQ_MAX; ++i) qa.q[i] = i < n_q ? q[i] : 0.0;
  for (int i = 0; i < n_q; ++i)
    if (!(qa.q[i] >= 0.0 && qa.q[i] <= 1.0)) return fail(SIMPLYP_EINVAL, "nanquantile: quantiles must lie in [0, 1]%s");
  if (simplyp_device_count() <= 0) return fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
  const int64_t need = simplyp_nanquantile_workspace_bytes(n_rows, n_cols);
  if (need > 0 && (!workspace || workspace_bytes < need))
    return fail(SIMPLYP_EINVAL, "nanquantile: workspace smaller than simplyp_nanquantile_workspace_bytes%s");
  if (n_rows == 0) return SIMPLYP_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (need == 0) {
    const size_t smem = (size_t)n_cols * sizeof(uint64_t);
    if (smem > 48 * 1024)
      SP_CUDA(cudaFuncSetAttribute(nanquantile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nanquantile_kernel<<<(unsigned)n_rows, NQ_THREADS, smem, st>>>(x, n_rows, n_cols, qa, quantiles, mean, count);
    g_launches.fetch_add(1);
    SP_CUDA(cudaGetLastError());
    return SIMPLYP_OK;
  }
  const long long per_block = (long long)NQ_HIST_THREADS * NQ_HIST_PER_THREAD;
  const long long slices = (n_cols + per_block - 1) / per_block;
  if (slices > 65535) return fail(SIMPLYP_EINVAL, "nanquantile: rows of at most 65535 * 4096 entries%s");
  NqRow* ws = static_cast<NqRow*>(workspace);
  nq_prepare_kernel<<<(unsigned)n_rows, NQ_THREADS, 0, st>>>(x, n_cols, qa, ws, mean, count);
  g_launches.fetch_add(1);
  SP_CUDA(cudaGetLastError());
  const dim3 hgrid((unsigned)n_rows, (unsigned)slices);
  for (int pass = 0; pass < 8; ++pass) {
    nq_hist_kernel<<<hgrid, NQ_HIST_THREADS, 0, st>>>(x, n_cols, n_q, pass, ws);
    nq_pick_kernel<<<(unsigned)n_rows, NQ_RANKS, 0, st>>>(n_rows, qa, pass, ws, quantiles);
    g_launches.fetch_add(2);
    SP_CUDA(cudaGetLastError());
  }
  return SIMPLYP_OK;
}

void simplyp_release_cache(void) {
  int n = 0, prev = -1;
  if (cudaGetDeviceCount(&n) != cudaSuccess) n = 0;
  cudaGetDevice(&prev);
  for (int d = 0; d < MAX_DEVICES; ++d) {
    HostCache& c = g_cache[d];
    std::lock_guard<std::mutex> guard(c.lock);
    if (!c.stream && !c.buf[0] && !c.epoch_flags) continue;
    if (d < n) cudaSetDevice(d);
    for (int i = 0; i < 8; ++i) {
      if (c.buf[i]) cudaFree(c.buf[i]);
      c.buf[i] = nullptr;
      c.cap[i] = 0;
    }
    if (c.stream) cudaStreamDestroy(c.stream);
    c.stream = nullptr;
    if (c.copy_stream) cudaStreamDestroy(c.copy_stream);
    c.copy_stream = nullptr;
    if (c.epoch_flags) cudaFreeHost(c.epoch_flags);
    c.epoch_flags = nullptr;
    c.epoch_flags_dev = nullptr;
  }
  if (prev >= 0) cudaSetDevice(prev);
  std::lock_guard<std::mutex> lock(g_topo_mutex);
  for (TopoImage& t : g_topo_images) cudaFreeHost(t.host);
  g_topo_images.clear();
}

int64_t simplyp_launch_count(void) { return g_launches.load(); }

double simplyp_measure_fp64_latency(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
    fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
    return -1.0;
  }
  cudaSetDevice(device);
  double* sink = nullptr;
  long long* cyc = nullptr;
  if (cudaMalloc(&sink, 8) != cudaSuccess || cudaMalloc(&cyc, 8) != cudaSuccess) return -1.0;
  const int iters = 4096;
  long long h = 0;
  for (int r = 0; r < 2; ++r) {
    fp64_latency_kernel<<<1, 32>>>(sink, cyc, iters, 0.999999, 1e-9);
    cudaMemcpy(&h, cyc, 8, cudaMemcpyDeviceToHost);
  }
  g_launches.fetch_add(2);
  cudaFree(sink);
  cudaFree(cyc);
  return (double)h / (16.0 * iters);
}

double simplyp_measure_fp64_peak(int device, int repeats) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
    fail(SIMPLYP_ENODEVICE, "no CUDA device%s");
    return -1.0;
  }
  cudaSetDevice(device);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  double* sink = nullptr;
  if (cudaMalloc(&sink, 8) != cudaSuccess) return -1.0;
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  fp64_peak_kernel<<<blocks, threads>>>(sink, 64, 0.999999, 1e-9);   // warm-up
  cudaDeviceSynchronize();
  double best = 0.0;
  for (int r = 0; r < (repeats > 0 ? repeats : 3); ++r) {
    cudaEventRecord(e0);
    fp64_peak_kernel<<<blocks, threads>>>(sink, iters, 0.999999, 1e-9);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = 2.0 * 64.0 * iters * (double)blocks * threads;
    const double tf = flops / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  g_launches.fetch_add(1 + (repeats > 0 ? repeats : 3));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sink);
  return best;
}

}  // extern "C"
