/*
 * simplyp_b200 — C-ABI of the B200-native SimplyP daily mass-balance integrator.
 *
 * This is the drop-in boundary for ONE path of the reference (JoeyYHT/SimplyP, v0-2A):
 * the body of run_simply_p's sub-catchment x day loop,
 *     Current_Release/v0-2A/simplyP/model.py:365-724
 * i.e. per (sub-catchment, day): forcing fetch (:497-501), upstream reach sums (:508-544),
 * erodibility (:549-594), EPC0 (:600-611), the scipy.integrate.odeint(ode_f, ...) call (:640,
 * RHS ode_f :58-187, gate f_x :23-37), state carry + groundwater floor (:643-670), the
 * discretised soil-P update (:684-715, discretized_soilP :39-56) and the 12+13 raw output columns
 * (:644, :721-724); plus, for calibration ensembles, the goodness-of-fit reductions of
 * visualise_results.py:441-449 and the Gaussian log-likelihood of Development/2016/MCMC.ipynb:213-242.
 *
 * The reference has no FFI of its own (it is pure Python; its only native code is SciPy's LSODA,
 * reached through a per-day Python callback).  The binding a maintainer adds is the ctypes stub
 * shown in INTEGRATION.md; simplyp_b200/_cabi.py is that stub.
 *
 * Conventions
 *  - plain C, no torch/STL types; all arrays are dense, row-major, IEEE fp64 unless stated;
 *  - "_device" entry points take DEVICE pointers owned by the caller and enqueue on `stream`
 *    (a cudaStream_t passed as void*; NULL = legacy default stream) without synchronising, so they can be
 *    overlapped with copies and captured into a CUDA graph (the host-side topology arrays are copied into
 *    pinned images the library keeps until simplyp_release_cache(); a call with a topology it has not seen
 *    allocates such an image, so issue one ordinary call before capturing in the strict capture mode);
 *  - "_host" entry points take HOST pointers, copy H2D, run, copy D2H and synchronise
 *    (this is what a reference-side caller that holds numpy arrays uses); their device buffers are cached
 *    PER DEVICE behind a per-device lock: one host thread per device runs concurrently with the others;
 *  - every entry point returns 0 on success or a negative SIMPLYP_E* code and never throws;
 *    simplyp_last_error() gives the message of the calling thread's last failure;
 *  - there is NO CPU fallback: without a CUDA device every compute entry point returns
 *    SIMPLYP_ENODEVICE.
 */
#ifndef SIMPLYP_B200_H
#define SIMPLYP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIMPLYP_ABI_VERSION 4

/* error codes */
#define SIMPLYP_OK          0
#define SIMPLYP_EINVAL     -1   /* bad argument (null pointer, bad dims, bad topology order) */
#define SIMPLYP_ENODEVICE  -2   /* no usable CUDA device */
#define SIMPLYP_ECUDA      -3   /* CUDA runtime error (see simplyp_last_error) */
#define SIMPLYP_ENOMEM     -4   /* device allocation failed */

/* ---- layouts ------------------------------------------------------------------------------- */

/* Per-member parameter vector: member_params[M][SIMPLYP_NP_MEMBER].
 * Names are the reference's (sheet "Constant" -> p, sheet "LU" -> p_LU[class]). */
enum {
  SIMPLYP_P_F_QUICK = 0,   /* p['f_quick']        */
  SIMPLYP_P_ALPHA,         /* p['alpha']          */
  SIMPLYP_P_FC,            /* p['fc']             */
  SIMPLYP_P_BETA,          /* p['beta']           */
  SIMPLYP_P_T_G,           /* p['T_g']            */
  SIMPLYP_P_QG_MIN,        /* p['Qg_min']         */
  SIMPLYP_P_A_Q,           /* p['a_Q']            */
  SIMPLYP_P_B_Q,           /* p['b_Q']            */
  SIMPLYP_P_QR0_INIT,      /* p['Qr0_init']  m3/s */
  SIMPLYP_P_MSOIL_M2,      /* p['Msoil_m2']       */
  SIMPLYP_P_KF,            /* p['Kf'] (used unless run_mode_cal) */
  SIMPLYP_P_TDPG,          /* p['TDPg']           */
  SIMPLYP_P_F_TDP,         /* p['f_TDP']          */
  SIMPLYP_P_E_PP,          /* p['E_PP']           */
  SIMPLYP_P_E_M,           /* p['E_M']            */
  SIMPLYP_P_K_M,           /* p['k_M']            */
  SIMPLYP_P_D_MAXE_SPR,    /* p['d_maxE_spr']     */
  SIMPLYP_P_D_MAXE_AUT,    /* p['d_maxE_aut']     */
  SIMPLYP_P_TS_A,          /* p_LU['A']['T_s']    */
  SIMPLYP_P_TS_S,          /* p_LU['S']['T_s']    */
  SIMPLYP_P_SOILP_A,       /* p_LU['A']['SoilPconc'] */
  SIMPLYP_P_SOILP_S,       /* p_LU['S']['SoilPconc'] */
  SIMPLYP_P_PNET_A,        /* p_LU['A']['P_netInput']  */
  SIMPLYP_P_PNET_NC,       /* p_LU['NC']['P_netInput'] */
  SIMPLYP_P_EPC0_A,        /* p_LU['A']['EPC0_init_mgl'] */
  SIMPLYP_P_EPC0_S,        /* p_LU['S']['EPC0_init_mgl'] */
  SIMPLYP_P_CCOVER_A,      /* p_LU['A']['C_cover']  */
  SIMPLYP_P_CCOVER_S,
  SIMPLYP_P_CCOVER_IG,
  SIMPLYP_P_CMEAS_A,       /* p_LU['A']['C_measures'] */
  SIMPLYP_P_CMEAS_S,
  SIMPLYP_P_CMEAS_IG,
  SIMPLYP_P_ERR_M0,        /* likelihood error scale m for observed series kind 0 (Q) ... */
  SIMPLYP_P_ERR_M1,        /* SS  */
  SIMPLYP_P_ERR_M2,        /* TDP */
  SIMPLYP_P_ERR_M3,        /* PP  */
  SIMPLYP_P_ERR_M4,        /* TP  */
  SIMPLYP_P_ERR_M5,        /* SRP */
  SIMPLYP_P_D_SNOW_0,      /* p['D_snow_0']  (read only when SimplypOptions.snow_on_device) */
  SIMPLYP_P_F_DDSM,        /* p['f_DDSM']    (read only when SimplypOptions.snow_on_device) */
  SIMPLYP_NP_MEMBER = 40   /* row stride */
};

/* Per-sub-catchment parameter vector: sc_params[Msc][S][SIMPLYP_NP_SC], Msc = 1 (shared by all
 * members) or M (per member).  Names are the rows of the reference's sheet "SC_reach" -> p_SC. */
enum {
  SIMPLYP_SC_A_CATCH = 0, SIMPLYP_SC_F_AR, SIMPLYP_SC_F_IG, SIMPLYP_SC_F_S,
  SIMPLYP_SC_F_NC_AR, SIMPLYP_SC_F_NC_IG, SIMPLYP_SC_F_NC_S, SIMPLYP_SC_F_SPR,
  SIMPLYP_SC_S_AR, SIMPLYP_SC_S_IG, SIMPLYP_SC_S_SN, SIMPLYP_SC_L_REACH,
  SIMPLYP_SC_S_REACH, SIMPLYP_SC_TDPEFF,
  SIMPLYP_NP_SC = 16       /* row stride (2 spare) */
};

/* forcing[D][SIMPLYP_NF]: P (rain+melt, mm/d; met_df['P']), PET (mm/d), day of year (1..366), T_air.
 * With SimplypOptions.snow_on_device column 0 holds the raw met_df['Precipitation'] and column 3 met_df['T_air']
 * (degrees C); P is then formed per member by the degree-day snow recursion of inputs.py:159-210 with that
 * member's D_snow_0 and f_DDSM.  Otherwise column 3 is ignored. */
#define SIMPLYP_NF 4

/* Raw output row per (member, sub-catchment, day): out[M][S][D][SIMPLYP_NOUT].
 * Columns 0..11 are the reference's df_ODE columns (model.py:737-739), 12..24 its df_nonODE
 * columns (model.py:743-745), in the reference's order. */
enum {
  SIMPLYP_O_VSA = 0, SIMPLYP_O_VSS, SIMPLYP_O_VG, SIMPLYP_O_VR, SIMPLYP_O_QR_END, SIMPLYP_O_QR,
  SIMPLYP_O_MSUS_END, SIMPLYP_O_MSUS_FLUX, SIMPLYP_O_TDPR_END, SIMPLYP_O_TDP_FLUX,
  SIMPLYP_O_PPR_END, SIMPLYP_O_PP_FLUX,
  SIMPLYP_O_QQ, SIMPLYP_O_QSA, SIMPLYP_O_QSS, SIMPLYP_O_QG, SIMPLYP_O_CCOVER_A,
  SIMPLYP_O_EPC0_A, SIMPLYP_O_EPC0_NC, SIMPLYP_O_TDPS_A, SIMPLYP_O_PLAB_A, SIMPLYP_O_CONC_A,
  SIMPLYP_O_TDPS_NC, SIMPLYP_O_PLAB_NC, SIMPLYP_O_CONC_NC,
  SIMPLYP_NOUT = 25
};

/* Observed series kinds (visualise_results.py:401,412-413): simulated counterpart in brackets */
enum {
  SIMPLYP_V_Q = 0,   /* Q_cumecs  */
  SIMPLYP_V_SS,      /* SS_mgl    */
  SIMPLYP_V_TDP,     /* TDP_mgl   */
  SIMPLYP_V_PP,      /* PP_mgl    */
  SIMPLYP_V_TP,      /* TP_mgl    */
  SIMPLYP_V_SRP,     /* SRP_mgl   */
  SIMPLYP_NVARKIND
};

/* Fit statistics per (member, observed series): stats[M][V][SIMPLYP_NSTAT] */
enum {
  SIMPLYP_ST_N = 0,      /* number of (obs, sim) pairs used                               */
  SIMPLYP_ST_NSE,        /* 1 - sum((o-s)^2)/sum((o-mean o)^2)       visualise_results.py:441 */
  SIMPLYP_ST_LOG_NSE,    /* same on natural logs                      :442-443             */
  SIMPLYP_ST_LOGLIK,     /* sum log N(o; s, (m s)^2)                  MCMC.ipynb:233-242   */
  SIMPLYP_ST_R2,         /* squared Pearson correlation               :446-447             */
  SIMPLYP_ST_PBIAS,      /* 100 sum(s-o)/sum(o)                       :448                 */
  SIMPLYP_ST_NRMSD,      /* 100 mean|s-o| / std(o) (population std)   :449                 */
  SIMPLYP_ST_SSE,        /* sum((o-s)^2)                                                   */
  SIMPLYP_ST_SPEARMAN,   /* Spearman's rank correlation (average ranks for ties)  :444-445 ; NaN unless
                            SimplypOptions.rank_stats is set                                    */
  SIMPLYP_ST_RESERVED,
  SIMPLYP_NSTAT          /* = 10 */
};

/* Integrator diagnostics per (member, sub-catchment): diag[M][S][SIMPLYP_NDIAG] (int64) */
enum {
  SIMPLYP_DG_STEPS = 0,  /* accepted + rejected step attempts      */
  SIMPLYP_DG_REJECTED,   /* rejected attempts                      */
  SIMPLYP_DG_RHS,        /* right-hand-side evaluations            */
  SIMPLYP_DG_STATUS,     /* bit 0: max steps/day hit, bit 1: non-finite state, bit 2: input wait timed out */
  SIMPLYP_NDIAG
};

typedef struct SimplypDims {
  int32_t n_members;       /* M  */
  int32_t n_sc;            /* S  */
  int32_t n_days;          /* D  */
  int32_t n_sc_param_sets; /* 1 or M */
  int32_t n_obs_series;    /* V (0 for simplyp_run) */
  int32_t reserved[3];
} SimplypDims;

typedef struct SimplypOptions {
  double  rtol;              /* relative tolerance of the embedded RK error control (of a day whose reach relaxes slowly:
                                both tolerances grow with the reach's rate constant, see INTEGRATION.md section 5) */
  double  atol;              /* absolute tolerance (same for all 12 states, like odeint's scalar atol) */
  double  step_len;          /* length of one forcing step in days (reference default 1.0) */
  int32_t max_steps_per_day; /* step attempts allowed per day before the status bit is raised */
  int32_t dynamic_epc0;      /* dynamic_options['Dynamic_EPC0'] == 'y' */
  int32_t dynamic_erodibility; /* dynamic_options['Dynamic_erodibility'] == 'y' */
  int32_t run_mode_cal;      /* p_SU.run_mode == 'cal': Kf derived per SC (model.py:449-451) */
  int32_t sc_qr0;            /* 0-based index of p['SC_Qr0'] in the run order */
  int32_t strict_quirks;     /* 1: replicate the leaked NC_type of model.py:442,676 */
  int32_t threads_per_block; /* reserved (0) */
  int32_t lanes_per_item;    /* lanes that integrate one (member, sub-catchment): 0 (default) or 4 — the quad kernel;
                                the round-1 one-thread-per-item kernel (1) was retired and is refused */
  int32_t pilot_days;        /* ensembles of one sub-catchment: the first `pilot_days` days are integrated in member
                                order by a pilot launch whose step counts order the members over the lock-step warps;
                                the main launch continues from its midnight state (0 = default 8, < 0 = no pilot;
                                the results do not depend on it) */
  int32_t rank_stats;        /* calibration: also reduce Spearman's r (stores the simulated value of every observed
                                day, M*V*D*8 bytes of workspace, and ranks them on the device afterwards) */
  int32_t snow_on_device;    /* 1: snow_hydrol_inputs (inputs.py:159-210) runs per member on the device (see forcing) */
  int32_t reserved[1];
} SimplypOptions;

/* ---- entry points -------------------------------------------------------------------------- */

int         simplyp_abi_version(void);
const char* simplyp_version(void);
const char* simplyp_last_error(void);
int         simplyp_device_count(void);
void        simplyp_default_options(SimplypOptions* opt);

/* Reach topology: sub-catchments are indexed 0..S-1 in RUN ORDER, which must be upstream-first
 * (model.py:524 raises KeyError otherwise).  parent_offsets[S+1], parent_ids[E] is the CSR list of
 * directly-upstream sub-catchments of each one (p_struc['Upstream_SCs'], model.py:480-487).
 * Writes levels[S] (0 = headwater).  Returns the number of levels or a negative error code. */
int simplyp_topology_levels(int32_t n_sc, const int32_t* parent_offsets, const int32_t* parent_ids,
                            int32_t* levels);

/* Bytes of device workspace simplyp_*_device needs for these dims (flux exchange, flags, cost ordering).
 * `calibrate`: 0 = simplyp_run_device, 1 = simplyp_calibrate_device, 3 = simplyp_calibrate_device with
 * SimplypOptions.rank_stats set.  dims->reserved[0] must hold the number of edges of the reach topology. */
int64_t simplyp_workspace_bytes(const SimplypDims* dims, int calibrate);

/* Full-output integration (replaces model.py:365-724 for every member):
 *   forcing[D][4], member_params[M][40], sc_params[Msc][S][16], CSR topology,
 *   out[M][S][D][25], diag[M][S][4] (may be NULL), workspace (may be NULL if S == 1). */
int simplyp_run_device(const SimplypDims* dims, const SimplypOptions* opt,
                       const double* forcing, const double* member_params, const double* sc_params,
                       const int32_t* parent_offsets, const int32_t* parent_ids,
                       double* out, int64_t* diag, void* workspace, void* stream);

/* Calibration mode: same integration, nothing written per day; instead fit statistics against
 * observed series are reduced on the fly.
 *   obs[V][D]     : observed value or NaN, aligned with forcing days
 *   obs_desc[V][2]: (sub-catchment index 0..S-1, series kind SIMPLYP_V_*); simplyp_calibrate_host refuses any other
 *                   row with SIMPLYP_EINVAL before device work.  The _device entry points take valid rows as a
 *                   precondition: checking rows in device memory would need a synchronising copy, which breaks
 *                   graph capture.  An invalid row there gives undefined statistics for that series.
 *   stats[M][V][SIMPLYP_NSTAT] */
int simplyp_calibrate_device(const SimplypDims* dims, const SimplypOptions* opt,
                             const double* forcing, const double* member_params, const double* sc_params,
                             const int32_t* parent_offsets, const int32_t* parent_ids,
                             const double* obs, const int32_t* obs_desc,
                             double* stats, int64_t* diag, void* workspace, void* stream);

/* Calibration mode fused with the all-gather of the statistics over peer memory (one process per GPU, NVLink /
 * NVSwitch): every rank integrates members [member_offset, member_offset + dims->n_members) of an ensemble of
 * n_members_total and its kernel stores each finished member's statistics straight into EVERY rank's gather buffer
 * (peer stores), so that the only thing left after the integration is a flag exchange: the rank raises `step` in
 * every peer's flag array and waits until every peer has raised it in its own (one small kernel, enqueued on `stream`).
 *   stats_bufs[r] : rank r's gather buffer [n_members_total][V][SIMPLYP_NSTAT] as mapped into THIS process
 *                   (own: an ordinary device pointer; peers: simplyp_ipc_import of their simplyp_ipc_export handle)
 *   flag_bufs[r]  : rank r's flags int32[SIMPLYP_MAX_RANKS], zero before the first call; flag_bufs[r][q] = last step
 *                   rank q has finished
 *   step          : strictly increasing from call to call, the same on all ranks.  A caller that reuses the buffers
 *                   alternates between two sets (a fast rank writes step k+1 while a slow one still reads step k).
 * The caller's `stats` argument is replaced by stats_bufs[rank] + member_offset rows.  SimplypOptions.rank_stats must
 * be 0 (Spearman's r is filled by a later kernel).  After the flag kernel, diag status bit 8 (on member 0, series 0 of
 * this rank) reports a peer that did not answer within ~2 s.  Replaces, on this path, torch.distributed's
 * all_gather_into_tensor (the reference has no multi-process form: Development/2016/MCMC.ipynb:29-31,380 uses an
 * IPython.parallel pool). */
#define SIMPLYP_MAX_RANKS 8
typedef struct {
  int32_t  n_ranks, rank;
  int64_t  member_offset, n_members_total;
  int64_t  step;
  double*  stats_bufs[SIMPLYP_MAX_RANKS];
  int32_t* flag_bufs[SIMPLYP_MAX_RANKS];
} SimplypPeerGather;

int simplyp_calibrate_gather_device(const SimplypDims* dims, const SimplypOptions* opt,
                                    const double* forcing, const double* member_params, const double* sc_params,
                                    const int32_t* parent_offsets, const int32_t* parent_ids,
                                    const double* obs, const int32_t* obs_desc,
                                    const SimplypPeerGather* gather, int64_t* diag, void* workspace, void* stream);

/* Peer-visible device memory for the buffers above: a zeroed cudaMalloc allocation of its own (an IPC handle maps a
 * whole allocation), its 64-byte CUDA IPC handle, and the mapping of another process's handle into this one. */
int simplyp_peer_alloc(int64_t bytes, void** dptr);
int simplyp_peer_free(void* dptr);
int simplyp_ipc_export(const void* dptr, unsigned char handle[64]);
int simplyp_ipc_import(const unsigned char handle[64], void** dptr);
int simplyp_ipc_close(void* dptr);

/* sum_to_waterbody (model.py:851-900) on the raw output of simplyp_run_device, for every member and day:
 *   out[M][S][D][25], reaches[n_reaches] = run-order indices of the reaches with In_final_flux? == 1 (device),
 *   waterbody[M][D][SIMPLYP_NWB] = Q_cumecs, Msus_kg/day, TDP_kg/day, PP_kg/day, SS_mgl, TDP_mgl, PP_mgl,
 *                                  TP_mgl, TP_kg/day, SRP_mgl, SRP_kg/day  (:878-892, derived_P_species :840-845) */
#define SIMPLYP_NWB 11
int simplyp_sum_to_waterbody_device(const SimplypDims* dims, const double* out, const double* sc_params,
                                    const double* member_params, const int32_t* reaches, int32_t n_reaches,
                                    double* waterbody, void* stream);

/* daily_PET (inputs.py:232-312; Thornthwaite 1948 via :416-508) on the device, for a record of whole calendar
 * years starting on 1 January: t_air[d * t_stride] daily mean air temperature, month_start[n_months + 1] = day index
 * at which each calendar month starts (device), year_is_leap[n_months / 12] (device; bit 0 = leap year, bit 1 = the
 * year uses the leap-year daylight-hours table: the reference keeps that table for all years after its first leap
 * year, inputs.py:269-273 — pass 3 for a leap year and 2 for the later non-leap years to reproduce it, 0/3 per
 * year for the calendar-correct choice), latitude in degrees;
 * pet[d * pet_stride] receives mm/day (stride 4 writes column 1 of a forcing matrix in place when pet = forcing + 1). */
int simplyp_thornthwaite_pet_device(int32_t n_days, int32_t n_months, const double* t_air, int32_t t_stride,
                                    const int32_t* month_start, const int32_t* year_is_leap, double latitude_deg,
                                    double* pet, int32_t pet_stride, void* stream);

/* ---- ensemble MCMC over the fused log-likelihood -------------------------------------------------
 * The affine-invariant stretch move (Goodman & Weare 2010; emcee's EnsembleSampler with its default StretchMove)
 * with a uniform prior box, for the calibration the reference does with emcee in Development/2016/MCMC.ipynb.
 * The W walkers are two contiguous halves of W/2; one iteration is, for half 0 and then half 1:
 *   simplyp_mcmc_propose_device  -> the free columns of that half's member_params (and sc_params) rows;
 *   zero that half's diag, then simplyp_calibrate_device on that half's rows;
 *   simplyp_mcmc_accept_device   -> Metropolis-Hastings test, walkers / lp / accepted updated (half 1: chain slot
 *                                   stored when (t+1) % thin == 0, then the iteration counter t is incremented).
 * Random words: Philox4x32-10 keyed by the seed, counter (walker, t low word, t high word, block), block 0 = partner
 * and stretch factor, block 1 = acceptance; t lives in device memory, so one captured iteration replays unchanged.
 * A proposal outside the box is flagged and its rows get the walker's CURRENT values (the integrator never sees an
 * out-of-box parameter); the accept step rejects it from the flag.
 * lp of a member = sum over its series of stats[.][v][SIMPLYP_ST_LOGLIK], or -inf if a diag status word of the member
 * is non-zero; the box prior adds 0 inside. */
#define SIMPLYP_MCMC_MAX_FREE 64
enum {
  SIMPLYP_MCMC_MEMBER = 0,  /* member_params[.][index]                                   */
  SIMPLYP_MCMC_SC_ALL,      /* sc_params[.][s][index] for every sub-catchment s          */
  SIMPLYP_MCMC_SC_AT        /* sc_params[.][pos][index], pos = position in the run order */
};

typedef struct {
  int32_t kind, index, pos, reserved;
  double  lo, hi;           /* prior box, lo < hi, both finite */
} SimplypMcmcParam;

typedef struct {
  int32_t n_walkers;        /* W: even, >= 2 * n_free */
  int32_t n_free;           /* K: 1..SIMPLYP_MCMC_MAX_FREE */
  int32_t n_sc;             /* S of the calibration runs */
  int32_t n_obs_series;     /* V of the calibration runs */
  int32_t sc_per_member;    /* sc_params is [W][S][NP_SC] (required by the SC targets) rather than [1][S][NP_SC] */
  int32_t thin;             /* chain slot stored every `thin` iterations */
  uint64_t seed;            /* Philox key: (low word, high word) */
  double  stretch;          /* a > 1 (emcee's default 2) */
  SimplypMcmcParam param[SIMPLYP_MCMC_MAX_FREE];
} SimplypMcmc;

typedef struct {            /* device pointers */
  double*  walkers;         /* [W][K] current states */
  double*  lp;              /* [W] their log-probabilities */
  double*  proposals;       /* [W/2][K] proposals of the active half */
  double*  log_z;           /* [W/2] ln z of those proposals */
  int32_t* out_of_box;      /* [W/2] 1: proposal outside the box */
  int64_t* iteration;       /* [1] t, the iteration in progress */
  int64_t* accepted;        /* [W] accepted proposals per walker */
  double*  chain;           /* [n_saved][W][K] */
  double*  chain_lp;        /* [n_saved][W] */
  int64_t  n_saved;         /* slots of chain / chain_lp */
  int64_t  chain_base;      /* iteration t stores slot (t+1)/thin - 1 - chain_base (floor(t_start/thin) of the run) */
} SimplypMcmcState;

/* member_params [W][NP_MEMBER], sc_params [1 or W][S][NP_SC]: the ensemble's rows; half = 0 or 1. */
int simplyp_mcmc_propose_device(const SimplypMcmc* mc, const SimplypMcmcState* state, int half,
                                double* member_params, double* sc_params, void* stream);
/* stats [W/2][V][NSTAT] and diag [W/2][S][NDIAG]: what simplyp_calibrate_device wrote for the active half's rows. */
int simplyp_mcmc_accept_device(const SimplypMcmc* mc, const SimplypMcmcState* state, int half,
                               const double* stats, const int64_t* diag, void* stream);
/* lp [W] of the current walkers from one calibration run of all W rows: stats [W][V][NSTAT], diag [W][S][NDIAG]. */
int simplyp_mcmc_init_device(const SimplypMcmc* mc, const SimplypMcmcState* state, const double* stats,
                             const int64_t* diag, void* stream);

/* ---- posterior predictive bands -----------------------------------------------------------------------------------
 * Quantiles over an ensemble of the simulated series the fused statistics see (SIMPLYP_V_* kinds of a reach), with or
 * without the likelihood's error model N(o; s, (m s)^2), m = member_params[.][SIMPLYP_P_ERR_M0 + kind].
 *
 * simplyp_predictive_draws_device: for a chunk of M members (dims: M, S, D, Msc = 1 or M) of a full-output run,
 *   out[M][S][D][25], member_params[M][NP_MEMBER], sc_params[Msc][S][NP_SC], diag[M][S][NDIAG], and
 *   series_desc[n_series][2] = (run-order reach 0..S-1, kind 0..5) on the device (a device-side precondition, like
 *   obs_desc), writes draws[n_series][D][n_members_total] at columns member_offset .. member_offset + M - 1:
 *     y = sim                        (obs_error = 0)
 *     y = sim + (m sim) eps          (obs_error = 1; eps standard normal by Box-Muller from Philox4x32-10 keyed by
 *                                     `seed` with counter (member_offset + m, day, series, 2): a pure function of
 *                                     (seed, member, day, series), whatever the chunking)
 *   A member with a non-zero SIMPLYP_DG_STATUS word at any reach draws NaN everywhere.
 * simplyp_nanquantile_device: for every row of x[n_rows][n_cols], exactly np.nanquantile(row, q, method='linear')
 *   (NaNs dropped; an all-NaN row gives NaN) into quantiles[n_q][n_rows], the mean of the non-NaN entries into
 *   mean[n_rows] and their count into count[n_rows].  q[n_q] is a HOST array of values in [0, 1], n_q <= SIMPLYP_NQ_MAX,
 *   passed to the kernels by value.  Rows longer than one block's shared memory holds (about 29k entries on B200) need
 *   simplyp_nanquantile_workspace_bytes(n_rows, n_cols) bytes of device workspace (0 otherwise).
 * Both only enqueue work on `stream` (no allocation, no synchronisation), so they can be captured into a graph. */
#define SIMPLYP_NQ_MAX 16
int simplyp_predictive_draws_device(const SimplypDims* dims, const double* out, const double* member_params,
                                    const double* sc_params, const int64_t* diag, const int32_t* series_desc,
                                    int32_t n_series, double* draws, int64_t n_members_total, int64_t member_offset,
                                    int32_t obs_error, uint64_t seed, void* stream);
int64_t simplyp_nanquantile_workspace_bytes(int64_t n_rows, int64_t n_cols);
int simplyp_nanquantile_device(const double* x, int64_t n_rows, int64_t n_cols, const double* q, int32_t n_q,
                               double* quantiles, double* mean, int64_t* count, void* workspace,
                               int64_t workspace_bytes, void* stream);

/* ---- period aggregates ---------------------------------------------------------------------------------------------
 * Period means, loads and flow-weighted mean concentrations of an ensemble, per reach and into the receiving water
 * body (simplyp_periods.cuh).  For a chunk of M members (dims: M, S, D, Msc = 1 or M) of a full-output run,
 * out[M][S][D][25], member_params[M][NP_MEMBER], sc_params[Msc][S][NP_SC] and diag[M][S][NDIAG] on the device, writes
 * values[n_series * n_periods][n_members_total] (row v * n_periods + p) at columns member_offset .. member_offset +
 * M - 1.
 * HOST arrays, passed to the kernel by value:
 *   series_desc[n_series][3] = (target, kind, statistic): target a run-order reach 0..S-1 or SIMPLYP_PERIOD_WATERBODY
 *     (the reaches waterbody_reaches[n_waterbody_reaches], run order, summed as simplyp_sum_to_waterbody_device sums
 *     them), kind SIMPLYP_V_*, statistic
 *       SIMPLYP_PERIOD_MEAN  mean over the period's days of the daily value (a reach: the value the fit statistics see;
 *                            the water body: its Q_cumecs or concentration column),
 *       SIMPLYP_PERIOD_LOAD  sum of the daily flux in kg (Q: volume in m3 = sum of Q_cumecs * 86400),
 *       SIMPLYP_PERIOD_FWMC  sum of the flux / sum of Q_cumecs * 1000/86400 in mg/l (not for Q);
 *   period_bounds[n_periods][2] = first and last day (inclusive) of each period, 0 <= first <= last < D.
 * Every sum runs over the days in ascending order, one rounding per addition, so a value depends on neither the
 * chunking nor the launch.  A member with a non-zero SIMPLYP_DG_STATUS word at any reach gives NaN in every row.
 * Only enqueues work on `stream`, so it can be captured into a graph. */
#define SIMPLYP_PERIOD_MAX_SERIES 64
#define SIMPLYP_PERIOD_MAX_PERIODS 2048
#define SIMPLYP_PERIOD_MAX_REACHES 256
#define SIMPLYP_PERIOD_WATERBODY (-1)
enum { SIMPLYP_PERIOD_MEAN = 0, SIMPLYP_PERIOD_LOAD = 1, SIMPLYP_PERIOD_FWMC = 2 };
int simplyp_period_aggregates_device(const SimplypDims* dims, const double* out, const double* member_params,
                                     const double* sc_params, const int64_t* diag, const int32_t* series_desc,
                                     int32_t n_series, const int32_t* period_bounds, int32_t n_periods,
                                     const int32_t* waterbody_reaches, int32_t n_waterbody_reaches, double* values,
                                     int64_t n_members_total, int64_t member_offset, void* stream);

/* ---- Sobol' sensitivity indices over a Saltelli design ------------------------------------------------------------
 * SALib's sobol.sample / sobol.analyze on the device.  K free parameters (the sampler's targets and boxes,
 * SimplypMcmcParam), N = n_base samples, P = K + 2 design members a sample (2K + 2 with second order).
 *
 * simplyp_sobol_design_device: overwrites the target columns of the design members [member_offset, member_offset + n)
 *   of member_params [N P][NP_MEMBER] and sc_params [N P][S][NP_SC] (or [1][S][NP_SC] without SC targets); the other
 *   columns keep what the caller put there (the base vectors).  Member m = i P + slot takes Sobol' point skip + i of
 *   the unscrambled 2K-dimensional sequence (Joe-Kuo new-joe-kuo-6.21201, SciPy's qmc.Sobol(scramble=False, bits=32)):
 *   slot 0 = A (coordinates 0..K-1), slot 1+j = AB_j (A with column j from B = coordinates K..2K-1), slot K+1+j =
 *   BA_j (second order: B with column j from A), slot P-1 = B.  Value = lo + (hi - lo) u, each operation rounded.
 * simplyp_sobol_outputs_device: Y[n_rows][M] from the fused statistics of the design (stats [M][V][NSTAT], diag
 *   [M][S][NDIAG]); row r is stats[.][rows[r][0]][rows[r][1]], or the sampler's member lp when rows[r][1] = -1
 *   (rows[n_rows][2] int32 on the device).  A member with a non-zero status word gives NaN in every row.
 * simplyp_sobol_indices_device: per row of Y[n_rows][N P] (member-major, as the design), with sample i used when its
 *   P values are all finite (n used; n < 2 or a zero variance gives NaN indices), c the mean of the used values,
 *   a = A - c etc. and V the population variance of {a_i} u {b_i}:
 *     S1_j = mean(b (ab_j - a)) / V,  ST_j = mean((a - ab_j)^2) / (2 V),
 *     S2_jk = mean(ba_j ab_k - a b) / V - S1_j - S1_k  (j < k, second order; NaN elsewhere).
 *   Bootstrap: resample t < n_boot draws n used samples with replacement, draw k at position (w n) >> 32 with w word
 *   k mod 4 of Philox4x32-10 keyed by `seed`, counter (t, k / 4, 0, 3); c stays, V is recomputed;
 *   *_conf = conf_z * std(ddof 1) over the resamples (NaN with n_boot < 2).  Outputs: S1, ST, S1_conf, ST_conf
 *   [n_rows][K]; S2, S2_conf [n_rows][K][K] (second order only, else may be NULL); mean (c), var (V) [n_rows];
 *   n_used [n_rows].  Sums run in a fixed order: results are bitwise reproducible.  Needs
 *   simplyp_sobol_workspace_bytes(sb, n_rows) bytes of device workspace.
 * All three only enqueue work on `stream` (no allocation, no synchronisation), so they can be captured into a graph. */
typedef struct {
  int32_t n_free;           /* K: 1..SIMPLYP_MCMC_MAX_FREE */
  int32_t n_sc;             /* S of the design's runs */
  int32_t sc_per_member;    /* sc_params is [N P][S][NP_SC] (required by the SC targets) */
  int32_t second_order;     /* 0 or 1 */
  int64_t n_base;           /* N: a power of two >= 2 */
  int64_t skip;             /* first Sobol' point; skip + N <= 2^32 */
  SimplypMcmcParam param[SIMPLYP_MCMC_MAX_FREE];
} SimplypSobol;

int simplyp_sobol_design_device(const SimplypSobol* sb, int64_t member_offset, int64_t n_members,
                                double* member_params, double* sc_params, void* stream);
int simplyp_sobol_outputs_device(const double* stats, const int64_t* diag, int64_t n_members, int32_t n_obs_series,
                                 int32_t n_sc, const int32_t* rows, int32_t n_rows, double* y, void* stream);
int64_t simplyp_sobol_workspace_bytes(const SimplypSobol* sb, int64_t n_rows);
int simplyp_sobol_indices_device(const SimplypSobol* sb, const double* y, int64_t n_rows, int32_t n_boot,
                                 double conf_z, uint64_t seed, double* S1, double* ST, double* S1_conf,
                                 double* ST_conf, double* S2, double* S2_conf, double* mean, double* var,
                                 int64_t* n_used, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- differential evolution ---------------------------------------------------------------------------------------
 * scipy.optimize.differential_evolution(updating='deferred', polish=False) over the fit statistics: the best parameter
 * set of K free parameters (the sampler's targets and boxes, SimplypMcmcParam) in a population of N members.  The
 * population lives in the unit cube; member rows get lo/hi-clamped values arg1 + (u - 0.5) arg2.  One generation is:
 *   simplyp_de_trial_device   -> trial[N][K] and the target columns of member_params (and sc_params) rows;
 *   zero diag, simplyp_calibrate_device on all N rows, simplyp_sobol_outputs_device -> y[R][N];
 *   simplyp_de_select_device  -> E = -sum_r weights[r] y[r][m] (+inf for a non-zero status word or a NaN), a trial
 *                                replaces its target when E_trial <= E_target; then one block reduces, in a fixed
 *                                order, the best index (lowest among the minimal energies), the mean and population
 *                                std of the finite energies and the counts; writes history row g + 1 - history_base =
 *                                (-E_best, -mean, std, replaced); adds the failed evaluations (E = +inf) to n_failed;
 *                                increments the generation g; sets converged = 1 and converged_at = g + 1 when every
 *                                energy is finite and std <= tol_abs + tol |mean|.
 * Once converged is set, trial and select return at once: replays queued after convergence change nothing.
 * simplyp_de_init_device: energies, best, history row 0 and n_failed from the evaluation of the population (the
 *   caller wrote its rows), converged = 0.
 * Random words: Philox4x32-10 keyed by the seed; member i at generation g takes group q of four words from counter
 * (i, g lo, g hi, 4 + 256 q), the generation's mutation factor F ~ U(mutation_lo, mutation_hi) from counter
 * (0xFFFFFFFF, g lo, g hi, 4); the word assignment is documented in csrc/simplyp_de.cuh.
 * All three only enqueue work on `stream` (no allocation, no synchronisation), so they can be captured into a graph. */
enum {
  SIMPLYP_DE_BEST1BIN = 0,  /* b' = x_best + F (x_r0 - x_r1) */
  SIMPLYP_DE_RAND1BIN       /* b' = x_r0 + F (x_r1 - x_r2)   */
};

typedef struct {
  int32_t n_population;     /* N: >= 3 (best1bin) or >= 4 (rand1bin), < 2^31 */
  int32_t n_free;           /* K: 1..SIMPLYP_MCMC_MAX_FREE */
  int32_t n_sc;             /* S of the calibration runs */
  int32_t sc_per_member;    /* sc_params is [N][S][NP_SC] (required by the SC targets) */
  int32_t strategy;         /* SIMPLYP_DE_BEST1BIN or SIMPLYP_DE_RAND1BIN */
  int32_t n_rows;           /* R objective rows of y, 1..65535 */
  uint64_t seed;            /* Philox key: (low word, high word) */
  double  mutation_lo, mutation_hi;   /* 0 <= lo <= hi < 2 */
  double  recombination;    /* CR in [0, 1] */
  double  tol, tol_abs;     /* finite, >= 0 */
  SimplypMcmcParam param[SIMPLYP_MCMC_MAX_FREE];
} SimplypDe;

typedef struct {            /* device pointers */
  double*  population;      /* [N][K] unit cube */
  double*  energy;          /* [N] */
  double*  trial;           /* [N][K] unit cube */
  int32_t* flags;           /* [N] bit 0: trial accepted, bit 1: evaluation failed */
  const double* weights;    /* [R] */
  int64_t* generation;      /* [1] g, generations completed */
  int64_t* best;            /* [1] index of the best member */
  int64_t* converged;       /* [1] 0 or 1 */
  int64_t* converged_at;    /* [1] generation at which converged was set */
  int64_t* n_failed;        /* [1] evaluations with E = +inf */
  double*  history;         /* [n_history][4] */
  int64_t  n_history;
  int64_t  history_base;    /* generation g + 1 ends in row g + 1 - history_base; the init writes row 0 */
} SimplypDeState;

/* member_params [N][NP_MEMBER], sc_params [1 or N][S][NP_SC]: the population's rows. */
int simplyp_de_trial_device(const SimplypDe* de, const SimplypDeState* state, double* member_params,
                            double* sc_params, void* stream);
/* y [R][N] (simplyp_sobol_outputs_device) and diag [N][S][NDIAG] of the evaluation of the trials. */
int simplyp_de_select_device(const SimplypDe* de, const SimplypDeState* state, const double* y, const int64_t* diag,
                             void* stream);
/* y [R][N] and diag [N][S][NDIAG] of the evaluation of the population. */
int simplyp_de_init_device(const SimplypDe* de, const SimplypDeState* state, const double* y, const int64_t* diag,
                           void* stream);

/* Host-buffer forms: same arguments as HOST pointers; the library stages them through its own
 * (cached) device buffers on `device`, runs and copies the result back before returning. */
int simplyp_run_host(int device, const SimplypDims* dims, const SimplypOptions* opt,
                     const double* forcing, const double* member_params, const double* sc_params,
                     const int32_t* parent_offsets, const int32_t* parent_ids,
                     double* out, int64_t* diag);

int simplyp_calibrate_host(int device, const SimplypDims* dims, const SimplypOptions* opt,
                           const double* forcing, const double* member_params, const double* sc_params,
                           const int32_t* parent_offsets, const int32_t* parent_ids,
                           const double* obs, const int32_t* obs_desc,
                           double* stats, int64_t* diag);

/* Releases the device buffers cached by the _host entry points (all devices) and the pinned topology images. */
void simplyp_release_cache(void);

/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t simplyp_launch_count(void);

/* Measures dependent-free DFMA throughput on `device` (TFLOP/s, 2 flop per FMA): the FP64
 * roofline denominator MEASURED_PEAKS.json does not carry.  Returns <0 on error. */
double simplyp_measure_fp64_peak(int device, int repeats);

/* Cycles per DEPENDENT DFMA (one warp, one chain): the fp64 pipeline latency that bounds a
 * single thread's progress when the ensemble is too small to fill the machine. */
double simplyp_measure_fp64_latency(int device);

#ifdef __cplusplus
}
#endif
#endif /* SIMPLYP_B200_H */
