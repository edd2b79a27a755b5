"""ctypes binding of ``libsimplyp_b200.so`` (``include/simplyp_b200.h``).

This is the stub a maintainer of the reference would add to call the CUDA path from Python (see
``INTEGRATION.md``).  There is no CPU fallback: if the shared library is missing, or no CUDA device
is visible, the compute entry points raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import packing as pk

_HERE = os.path.dirname(os.path.abspath(__file__))
# SIMPLYP_B200_LIB lets a developer A/B-test another build of the same library (still CUDA-only).
LIB_PATH = os.environ.get("SIMPLYP_B200_LIB") or os.path.join(_HERE, "lib", "libsimplyp_b200.so")

EXPORTS = [
    "simplyp_abi_version", "simplyp_version", "simplyp_last_error", "simplyp_device_count",
    "simplyp_default_options", "simplyp_topology_levels", "simplyp_workspace_bytes",
    "simplyp_run_device", "simplyp_calibrate_device", "simplyp_run_host", "simplyp_calibrate_host",
    "simplyp_release_cache", "simplyp_launch_count", "simplyp_measure_fp64_peak",
    "simplyp_measure_fp64_latency", "simplyp_sum_to_waterbody_device", "simplyp_thornthwaite_pet_device",
    "simplyp_calibrate_gather_device", "simplyp_peer_alloc", "simplyp_peer_free", "simplyp_ipc_export",
    "simplyp_ipc_import", "simplyp_ipc_close", "simplyp_mcmc_propose_device", "simplyp_mcmc_accept_device",
    "simplyp_mcmc_init_device", "simplyp_predictive_draws_device", "simplyp_nanquantile_workspace_bytes",
    "simplyp_nanquantile_device", "simplyp_sobol_design_device", "simplyp_sobol_outputs_device",
    "simplyp_sobol_workspace_bytes", "simplyp_sobol_indices_device", "simplyp_de_trial_device",
    "simplyp_de_select_device", "simplyp_de_init_device", "simplyp_period_aggregates_device",
    "simplyp_calibrate_ar1_device", "simplyp_de_scale_device", "simplyp_nsga2_workspace_bytes",
    "simplyp_nsga2_init_device", "simplyp_nsga2_offspring_device", "simplyp_nsga2_survive_device",
    "simplyp_morris_workspace_bytes", "simplyp_morris_select_device", "simplyp_morris_design_device",
    "simplyp_morris_effects_device",
]
MAX_RANKS = 8


class SimplypDims(C.Structure):
    _fields_ = [("n_members", C.c_int32), ("n_sc", C.c_int32), ("n_days", C.c_int32),
                ("n_sc_param_sets", C.c_int32), ("n_obs_series", C.c_int32), ("reserved", C.c_int32 * 3)]


class SimplypOptions(C.Structure):
    _fields_ = [("rtol", C.c_double), ("atol", C.c_double), ("step_len", C.c_double),
                ("max_steps_per_day", C.c_int32), ("dynamic_epc0", C.c_int32),
                ("dynamic_erodibility", C.c_int32), ("run_mode_cal", C.c_int32), ("sc_qr0", C.c_int32),
                ("strict_quirks", C.c_int32), ("threads_per_block", C.c_int32), ("lanes_per_item", C.c_int32),
                ("pilot_days", C.c_int32), ("rank_stats", C.c_int32), ("snow_on_device", C.c_int32), ("reserved", C.c_int32 * 1)]


class SimplypPeerGather(C.Structure):
    _fields_ = [("n_ranks", C.c_int32), ("rank", C.c_int32), ("member_offset", C.c_int64),
                ("n_members_total", C.c_int64), ("step", C.c_int64), ("stats_bufs", C.c_void_p * MAX_RANKS),
                ("flag_bufs", C.c_void_p * MAX_RANKS)]


MCMC_MAX_FREE = 64
NQ_MAX = 16
PERIOD_MAX_SERIES, PERIOD_MAX_PERIODS, PERIOD_MAX_REACHES = 64, 2048, 256
PERIOD_WATERBODY = -1
PERIOD_STATS = {"mean": 0, "load": 1, "fwmc": 2}
MCMC_MEMBER, MCMC_SC_ALL, MCMC_SC_AT, MCMC_ERROR_MODEL = 0, 1, 2, 3
AR1_MAX_SERIES = 64
DE_STRATEGIES = {"best1bin": 0, "rand1bin": 1}
NSGA2_MAX_OBJECTIVES = 16
MORRIS_MAX_CANDIDATES = 8192


class SimplypMcmcParam(C.Structure):
    _fields_ = [("kind", C.c_int32), ("index", C.c_int32), ("pos", C.c_int32), ("reserved", C.c_int32),
                ("lo", C.c_double), ("hi", C.c_double)]


class SimplypMcmc(C.Structure):
    _fields_ = [("n_walkers", C.c_int32), ("n_free", C.c_int32), ("n_sc", C.c_int32), ("n_obs_series", C.c_int32),
                ("sc_per_member", C.c_int32), ("thin", C.c_int32), ("seed", C.c_uint64), ("stretch", C.c_double),
                ("param", SimplypMcmcParam * MCMC_MAX_FREE)]


class SimplypMcmcState(C.Structure):
    _fields_ = [("walkers", C.c_void_p), ("lp", C.c_void_p), ("proposals", C.c_void_p), ("log_z", C.c_void_p),
                ("out_of_box", C.c_void_p), ("iteration", C.c_void_p), ("accepted", C.c_void_p),
                ("chain", C.c_void_p), ("chain_lp", C.c_void_p), ("n_saved", C.c_int64), ("chain_base", C.c_int64)]


class SimplypSobol(C.Structure):
    _fields_ = [("n_free", C.c_int32), ("n_sc", C.c_int32), ("sc_per_member", C.c_int32), ("second_order", C.c_int32),
                ("n_base", C.c_int64), ("skip", C.c_int64), ("param", SimplypMcmcParam * MCMC_MAX_FREE)]


class SimplypMorris(C.Structure):
    _fields_ = [("n_free", C.c_int32), ("n_sc", C.c_int32), ("sc_per_member", C.c_int32), ("num_levels", C.c_int32),
                ("n_trajectories", C.c_int32), ("n_candidates", C.c_int32), ("seed", C.c_uint64),
                ("param", SimplypMcmcParam * MCMC_MAX_FREE)]


class SimplypDe(C.Structure):
    _fields_ = [("n_population", C.c_int32), ("n_free", C.c_int32), ("n_sc", C.c_int32), ("sc_per_member", C.c_int32),
                ("strategy", C.c_int32), ("n_rows", C.c_int32), ("seed", C.c_uint64), ("mutation_lo", C.c_double),
                ("mutation_hi", C.c_double), ("recombination", C.c_double), ("tol", C.c_double),
                ("tol_abs", C.c_double), ("param", SimplypMcmcParam * MCMC_MAX_FREE)]


class SimplypDeState(C.Structure):
    _fields_ = [("population", C.c_void_p), ("energy", C.c_void_p), ("trial", C.c_void_p), ("flags", C.c_void_p),
                ("weights", C.c_void_p), ("generation", C.c_void_p), ("best", C.c_void_p), ("converged", C.c_void_p),
                ("converged_at", C.c_void_p), ("n_failed", C.c_void_p), ("history", C.c_void_p),
                ("n_history", C.c_int64), ("history_base", C.c_int64)]


class SimplypNsga2(C.Structure):
    _fields_ = [("n_population", C.c_int32), ("n_free", C.c_int32), ("n_objectives", C.c_int32), ("n_sc", C.c_int32),
                ("sc_per_member", C.c_int32), ("reserved", C.c_int32), ("seed", C.c_uint64), ("crossover", C.c_double),
                ("mutation", C.c_double), ("eta_c", C.c_double), ("eta_m", C.c_double),
                ("sense", C.c_double * NSGA2_MAX_OBJECTIVES), ("param", SimplypMcmcParam * MCMC_MAX_FREE)]


class SimplypNsga2State(C.Structure):
    _fields_ = [("population", C.c_void_p), ("objectives", C.c_void_p), ("rank", C.c_void_p), ("crowding", C.c_void_p),
                ("offspring", C.c_void_p), ("generation", C.c_void_p), ("n_failed", C.c_void_p),
                ("history", C.c_void_p), ("n_history", C.c_int64), ("history_base", C.c_int64),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64)]


class SimplypAr1(C.Structure):
    _fields_ = [("phi", C.c_void_p), ("row_stride", C.c_int64), ("col", C.c_int32 * AR1_MAX_SERIES)]


class SimplypError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (built by ``__graft_entry__.build()``); raise if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SimplypError("%s not built — run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    dp, ip, lp, vp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.c_void_p
    lib.simplyp_abi_version.restype = C.c_int
    lib.simplyp_version.restype = C.c_char_p
    lib.simplyp_last_error.restype = C.c_char_p
    lib.simplyp_device_count.restype = C.c_int
    lib.simplyp_default_options.argtypes = [C.POINTER(SimplypOptions)]
    lib.simplyp_default_options.restype = None
    lib.simplyp_topology_levels.argtypes = [C.c_int32, ip, ip, ip]
    lib.simplyp_topology_levels.restype = C.c_int
    lib.simplyp_workspace_bytes.argtypes = [C.POINTER(SimplypDims), C.c_int]
    lib.simplyp_workspace_bytes.restype = C.c_int64
    lib.simplyp_run_device.argtypes = [C.POINTER(SimplypDims), C.POINTER(SimplypOptions), vp, vp, vp, ip, ip,
                                       vp, vp, vp, vp]
    lib.simplyp_run_device.restype = C.c_int
    lib.simplyp_calibrate_device.argtypes = [C.POINTER(SimplypDims), C.POINTER(SimplypOptions), vp, vp, vp, ip, ip,
                                             vp, vp, vp, vp, vp, vp]
    lib.simplyp_calibrate_device.restype = C.c_int
    lib.simplyp_run_host.argtypes = [C.c_int, C.POINTER(SimplypDims), C.POINTER(SimplypOptions), dp, dp, dp, ip, ip,
                                     dp, lp]
    lib.simplyp_run_host.restype = C.c_int
    lib.simplyp_calibrate_host.argtypes = [C.c_int, C.POINTER(SimplypDims), C.POINTER(SimplypOptions), dp, dp, dp,
                                           ip, ip, dp, ip, dp, lp]
    lib.simplyp_calibrate_host.restype = C.c_int
    lib.simplyp_release_cache.restype = None
    lib.simplyp_launch_count.restype = C.c_int64
    lib.simplyp_measure_fp64_peak.argtypes = [C.c_int, C.c_int]
    lib.simplyp_measure_fp64_peak.restype = C.c_double
    lib.simplyp_measure_fp64_latency.argtypes = [C.c_int]
    lib.simplyp_measure_fp64_latency.restype = C.c_double
    lib.simplyp_sum_to_waterbody_device.argtypes = [C.POINTER(SimplypDims), vp, vp, vp, vp, C.c_int32, vp, vp]
    lib.simplyp_sum_to_waterbody_device.restype = C.c_int
    lib.simplyp_thornthwaite_pet_device.argtypes = [C.c_int32, C.c_int32, vp, C.c_int32, vp, vp, C.c_double, vp,
                                                    C.c_int32, vp]
    lib.simplyp_thornthwaite_pet_device.restype = C.c_int
    lib.simplyp_calibrate_gather_device.argtypes = [C.POINTER(SimplypDims), C.POINTER(SimplypOptions), vp, vp, vp, ip,
                                                    ip, vp, vp, C.POINTER(SimplypPeerGather), vp, vp, vp]
    lib.simplyp_calibrate_gather_device.restype = C.c_int
    lib.simplyp_calibrate_ar1_device.argtypes = [C.POINTER(SimplypDims), C.POINTER(SimplypOptions), vp, vp, vp, ip, ip,
                                                 vp, vp, C.POINTER(SimplypAr1), vp, vp, vp, vp]
    lib.simplyp_calibrate_ar1_device.restype = C.c_int
    lib.simplyp_peer_alloc.argtypes = [C.c_int64, C.POINTER(C.c_void_p)]
    lib.simplyp_peer_alloc.restype = C.c_int
    lib.simplyp_peer_free.argtypes = [vp]
    lib.simplyp_peer_free.restype = C.c_int
    lib.simplyp_ipc_export.argtypes = [vp, C.c_char_p]
    lib.simplyp_ipc_export.restype = C.c_int
    lib.simplyp_ipc_import.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
    lib.simplyp_ipc_import.restype = C.c_int
    lib.simplyp_ipc_close.argtypes = [vp]
    lib.simplyp_ipc_close.restype = C.c_int
    mp, sp = C.POINTER(SimplypMcmc), C.POINTER(SimplypMcmcState)
    lib.simplyp_mcmc_propose_device.argtypes = [mp, sp, C.c_int, vp, vp, vp]
    lib.simplyp_mcmc_propose_device.restype = C.c_int
    lib.simplyp_mcmc_accept_device.argtypes = [mp, sp, C.c_int, vp, vp, vp]
    lib.simplyp_mcmc_accept_device.restype = C.c_int
    lib.simplyp_mcmc_init_device.argtypes = [mp, sp, vp, vp, vp]
    lib.simplyp_mcmc_init_device.restype = C.c_int
    lib.simplyp_predictive_draws_device.argtypes = [C.POINTER(SimplypDims), vp, vp, vp, vp, vp, C.c_int32, vp,
                                                    C.c_int64, C.c_int64, C.c_int32, C.c_uint64, vp]
    lib.simplyp_predictive_draws_device.restype = C.c_int
    lib.simplyp_period_aggregates_device.argtypes = [C.POINTER(SimplypDims), vp, vp, vp, vp, ip, C.c_int32, ip,
                                                     C.c_int32, ip, C.c_int32, vp, C.c_int64, C.c_int64, vp]
    lib.simplyp_period_aggregates_device.restype = C.c_int
    lib.simplyp_nanquantile_workspace_bytes.argtypes = [C.c_int64, C.c_int64]
    lib.simplyp_nanquantile_workspace_bytes.restype = C.c_int64
    lib.simplyp_nanquantile_device.argtypes = [vp, C.c_int64, C.c_int64, dp, C.c_int32, vp, vp, vp, vp, C.c_int64, vp]
    lib.simplyp_nanquantile_device.restype = C.c_int
    sbp = C.POINTER(SimplypSobol)
    lib.simplyp_sobol_design_device.argtypes = [sbp, C.c_int64, C.c_int64, vp, vp, vp]
    lib.simplyp_sobol_design_device.restype = C.c_int
    lib.simplyp_sobol_outputs_device.argtypes = [vp, vp, C.c_int64, C.c_int32, C.c_int32, vp, C.c_int32, vp, vp]
    lib.simplyp_sobol_outputs_device.restype = C.c_int
    lib.simplyp_sobol_workspace_bytes.argtypes = [sbp, C.c_int64]
    lib.simplyp_sobol_workspace_bytes.restype = C.c_int64
    lib.simplyp_sobol_indices_device.argtypes = [sbp, vp, C.c_int64, C.c_int32, C.c_double, C.c_uint64, vp, vp, vp,
                                                 vp, vp, vp, vp, vp, vp, vp, C.c_int64, vp]
    lib.simplyp_sobol_indices_device.restype = C.c_int
    dep, dsp = C.POINTER(SimplypDe), C.POINTER(SimplypDeState)
    lib.simplyp_de_trial_device.argtypes = [dep, dsp, vp, vp, vp]
    lib.simplyp_de_trial_device.restype = C.c_int
    lib.simplyp_de_select_device.argtypes = [dep, dsp, vp, vp, vp]
    lib.simplyp_de_select_device.restype = C.c_int
    lib.simplyp_de_init_device.argtypes = [dep, dsp, vp, vp, vp]
    lib.simplyp_de_init_device.restype = C.c_int
    lib.simplyp_de_scale_device.argtypes = [dep, vp, C.c_int64, vp, vp]
    lib.simplyp_de_scale_device.restype = C.c_int
    nsp, nssp = C.POINTER(SimplypNsga2), C.POINTER(SimplypNsga2State)
    lib.simplyp_nsga2_workspace_bytes.argtypes = [nsp]
    lib.simplyp_nsga2_workspace_bytes.restype = C.c_int64
    for name in ("simplyp_nsga2_init_device", "simplyp_nsga2_offspring_device", "simplyp_nsga2_survive_device"):
        getattr(lib, name).argtypes = [nsp, nssp, vp, vp, vp]
        getattr(lib, name).restype = C.c_int
    mop = C.POINTER(SimplypMorris)
    lib.simplyp_morris_workspace_bytes.argtypes = [mop, C.c_int64]
    lib.simplyp_morris_workspace_bytes.restype = C.c_int64
    lib.simplyp_morris_select_device.argtypes = [mop, vp, vp, C.c_int64, vp]
    lib.simplyp_morris_select_device.restype = C.c_int
    lib.simplyp_morris_design_device.argtypes = [mop, vp, C.c_int64, C.c_int64, vp, vp, vp]
    lib.simplyp_morris_design_device.restype = C.c_int
    lib.simplyp_morris_effects_device.argtypes = [mop, vp, vp, C.c_int64, C.c_int32, C.c_double, vp, vp, vp, vp, vp,
                                                  vp, C.c_int64, vp]
    lib.simplyp_morris_effects_device.restype = C.c_int
    if lib.simplyp_abi_version() != 4:
        raise SimplypError("ABI version mismatch")
    _lib = lib
    return lib


def _check(rc):
    if rc != 0:
        raise SimplypError("simplyp_b200 error %d: %s" % (rc, load().simplyp_last_error().decode()))


def require_device():
    lib = load()
    if lib.simplyp_device_count() <= 0:
        raise SimplypError("no CUDA device visible: simplyp_b200 has no CPU fallback")
    return lib


def default_options(**overrides):
    opt = SimplypOptions()
    load().simplyp_default_options(C.byref(opt))
    for k, v in overrides.items():
        if not hasattr(opt, k):
            raise AttributeError(k)
        setattr(opt, k, v)
    return opt


def make_dims(n_members, n_sc, n_days, n_sc_param_sets=1, n_obs_series=0, n_edges=0):
    d = SimplypDims()
    d.n_members, d.n_sc, d.n_days = int(n_members), int(n_sc), int(n_days)
    d.n_sc_param_sets, d.n_obs_series = int(n_sc_param_sets), int(n_obs_series)
    d.reserved[0] = int(n_edges)
    return d


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _iptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _c64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (shape, a.shape))
    return a


def _topology_arrays(parent_offsets, parent_ids):
    po = np.ascontiguousarray(parent_offsets, dtype=np.int32)
    pid = np.ascontiguousarray(parent_ids, dtype=np.int32)
    if pid.size == 0:
        pid = np.zeros(1, dtype=np.int32)
    return po, pid


def topology_levels(parent_offsets, parent_ids):
    po, pid = _topology_arrays(parent_offsets, parent_ids)
    S = len(po) - 1
    lv = np.zeros(max(S, 1), dtype=np.int32)
    n = load().simplyp_topology_levels(S, _iptr(po), _iptr(pid), _iptr(lv))
    if n < 0:
        _check(n)
    return n, lv[:S]


# ------------------------------------------------------------------------------------------ host-buffer calls
def _result_buffer(given, shape, dtype):
    """A caller-supplied result buffer (e.g. pinned host memory) must be C-contiguous with the expected shape/dtype."""
    if given is None:
        return np.zeros(shape, dtype=dtype) if dtype == np.int64 else np.empty(shape, dtype=dtype)
    if tuple(given.shape) != tuple(shape) or given.dtype != dtype or not given.flags["C_CONTIGUOUS"]:
        raise ValueError("result buffer must be a C-contiguous %s array of shape %s" % (np.dtype(dtype).name, tuple(shape)))
    return given


def run_host(forcing, member_params, sc_params, parent_offsets, parent_ids, opt, device=0, want_diag=True, out=None,
             diag=None):
    """numpy in / numpy out through ``simplyp_run_host``.  Returns (out [M][S][D][25], diag [M][S][4]); ``out`` /
    ``diag`` may be given (pinned host memory makes the copies asynchronous DMA)."""
    lib = require_device()
    forcing = _c64(forcing)
    member_params = _c64(member_params)
    sc_params = _c64(sc_params)
    if sc_params.ndim == 2:
        sc_params = sc_params[None]
    M, D = member_params.shape[0], forcing.shape[0]
    Msc, S = sc_params.shape[0], sc_params.shape[1]
    po, pid = _topology_arrays(parent_offsets, parent_ids)
    dims = make_dims(M, S, D, Msc, 0, int(po[-1]))
    out = _result_buffer(out, (M, S, D, pk.NOUT), np.float64)
    diag = _result_buffer(diag, (M, S, pk.NDIAG), np.int64)
    rc = lib.simplyp_run_host(device, C.byref(dims), C.byref(opt), _dptr(forcing), _dptr(member_params),
                              _dptr(sc_params), _iptr(po), _iptr(pid), _dptr(out),
                              diag.ctypes.data_as(C.POINTER(C.c_int64)) if want_diag else None)
    _check(rc)
    return out, diag


def calibrate_host(forcing, member_params, sc_params, parent_offsets, parent_ids, obs, obs_desc, opt,
                   device=0, want_diag=True, stats=None, diag=None):
    """numpy in / numpy out through ``simplyp_calibrate_host``.  Returns (stats [M][V][10], diag [M][S][4])."""
    lib = require_device()
    forcing = _c64(forcing)
    member_params = _c64(member_params)
    sc_params = _c64(sc_params)
    if sc_params.ndim == 2:
        sc_params = sc_params[None]
    obs = _c64(obs)
    obs_desc = np.ascontiguousarray(obs_desc, dtype=np.int32)
    M, D = member_params.shape[0], forcing.shape[0]
    Msc, S = sc_params.shape[0], sc_params.shape[1]
    V = obs.shape[0]
    po, pid = _topology_arrays(parent_offsets, parent_ids)
    dims = make_dims(M, S, D, Msc, V, int(po[-1]))
    stats = _result_buffer(stats, (M, V, pk.NSTAT), np.float64)
    diag = _result_buffer(diag, (M, S, pk.NDIAG), np.int64)
    rc = lib.simplyp_calibrate_host(device, C.byref(dims), C.byref(opt), _dptr(forcing), _dptr(member_params),
                                    _dptr(sc_params), _iptr(po), _iptr(pid), _dptr(obs), _iptr(obs_desc),
                                    _dptr(stats), diag.ctypes.data_as(C.POINTER(C.c_int64)) if want_diag else None)
    _check(rc)
    return stats, diag


# ------------------------------------------------------------------------------------------ device-pointer calls
def run_device(dims, opt, forcing_ptr, member_ptr, sc_ptr, parent_offsets, parent_ids, out_ptr, diag_ptr,
               ws_ptr, stream_ptr):
    """Raw device-pointer call (torch ``.data_ptr()`` integers); enqueues on ``stream_ptr``."""
    lib = require_device()
    po, pid = _topology_arrays(parent_offsets, parent_ids)
    _check(lib.simplyp_run_device(C.byref(dims), C.byref(opt), forcing_ptr, member_ptr, sc_ptr, _iptr(po), _iptr(pid),
                                  out_ptr, diag_ptr, ws_ptr, stream_ptr))


def calibrate_device(dims, opt, forcing_ptr, member_ptr, sc_ptr, parent_offsets, parent_ids, obs_ptr, desc_ptr,
                     stats_ptr, diag_ptr, ws_ptr, stream_ptr):
    lib = require_device()
    po, pid = _topology_arrays(parent_offsets, parent_ids)
    _check(lib.simplyp_calibrate_device(C.byref(dims), C.byref(opt), forcing_ptr, member_ptr, sc_ptr, _iptr(po),
                                        _iptr(pid), obs_ptr, desc_ptr, stats_ptr, diag_ptr, ws_ptr, stream_ptr))


def calibrate_gather_device(dims, opt, forcing_ptr, member_ptr, sc_ptr, parent_offsets, parent_ids, obs_ptr, desc_ptr,
                            gather, diag_ptr, ws_ptr, stream_ptr):
    """Calibration fused with the all-gather of the statistics over peer memory (``gather``: SimplypPeerGather)."""
    lib = require_device()
    po, pid = _topology_arrays(parent_offsets, parent_ids)
    _check(lib.simplyp_calibrate_gather_device(C.byref(dims), C.byref(opt), forcing_ptr, member_ptr, sc_ptr, _iptr(po),
                                               _iptr(pid), obs_ptr, desc_ptr, C.byref(gather), diag_ptr, ws_ptr,
                                               stream_ptr))


def make_ar1(phi_ptr, row_stride, col):
    """SimplypAr1: phi of member m, series v at ``phi_ptr`` (device) + (m * row_stride + col[v]) doubles; col[v] < 0
    keeps the iid likelihood of series v."""
    col = [int(c) for c in col]
    if len(col) > AR1_MAX_SERIES:
        raise ValueError("at most %d series with an AR(1) error model" % AR1_MAX_SERIES)
    ar = SimplypAr1()
    ar.phi, ar.row_stride = phi_ptr, int(row_stride)
    for v in range(AR1_MAX_SERIES):
        ar.col[v] = col[v] if v < len(col) else -1
    return ar


def calibrate_ar1_device(dims, opt, forcing_ptr, member_ptr, sc_ptr, parent_offsets, parent_ids, obs_ptr, desc_ptr,
                         ar1, stats_ptr, diag_ptr, ws_ptr, stream_ptr):
    """Calibration with the AR(1) error model of ``ar1`` (:func:`make_ar1`) in the log-likelihood."""
    lib = require_device()
    po, pid = _topology_arrays(parent_offsets, parent_ids)
    _check(lib.simplyp_calibrate_ar1_device(C.byref(dims), C.byref(opt), forcing_ptr, member_ptr, sc_ptr, _iptr(po),
                                            _iptr(pid), obs_ptr, desc_ptr, C.byref(ar1), stats_ptr, diag_ptr, ws_ptr,
                                            stream_ptr))


def peer_alloc(n_bytes):
    p = C.c_void_p()
    _check(require_device().simplyp_peer_alloc(int(n_bytes), C.byref(p)))
    return int(p.value)


def peer_free(ptr):
    _check(load().simplyp_peer_free(C.c_void_p(ptr)))


def ipc_export(ptr):
    buf = C.create_string_buffer(64)
    _check(load().simplyp_ipc_export(C.c_void_p(ptr), buf))
    return bytes(buf.raw)


def ipc_import(handle):
    p = C.c_void_p()
    _check(load().simplyp_ipc_import(C.create_string_buffer(bytes(handle), 64), C.byref(p)))
    return int(p.value)


def ipc_close(ptr):
    _check(load().simplyp_ipc_close(C.c_void_p(ptr)))


def sum_to_waterbody_device(dims, out_ptr, sc_ptr, member_ptr, reaches_ptr, n_reaches, wb_ptr, stream_ptr):
    lib = require_device()
    _check(lib.simplyp_sum_to_waterbody_device(C.byref(dims), out_ptr, sc_ptr, member_ptr, reaches_ptr,
                                               int(n_reaches), wb_ptr, stream_ptr))


def thornthwaite_pet_device(n_days, n_months, t_air_ptr, t_stride, month_start_ptr, year_is_leap_ptr, latitude_deg,
                            pet_ptr, pet_stride, stream_ptr):
    """Reference ``daily_PET`` (``inputs.py:232-312``) on device pointers; asynchronous on ``stream_ptr``."""
    _check(load().simplyp_thornthwaite_pet_device(int(n_days), int(n_months), C.c_void_p(t_air_ptr), int(t_stride),
                                                  C.c_void_p(month_start_ptr), C.c_void_p(year_is_leap_ptr),
                                                  float(latitude_deg), C.c_void_p(pet_ptr), int(pet_stride),
                                                  C.c_void_p(stream_ptr)))


def _u64(seed):
    """A seed as the uint64 the C-ABI takes (Python ints of any sign or size, modulo 2^64)."""
    return int(seed) & 0xFFFFFFFFFFFFFFFF


def _free_params(spec, targets, lo, hi):
    """``spec`` (SimplypMcmc, SimplypSobol, SimplypMorris, SimplypDe or SimplypNsga2) with ``n_free`` and ``param``
    set to the free parameters ``targets`` [(kind, index, pos)] (``MCMC_MEMBER`` / ``MCMC_SC_ALL`` / ``MCMC_SC_AT`` /
    ``MCMC_ERROR_MODEL``) and their boxes ``[lo[k], hi[k]]``."""
    if not 1 <= len(targets) <= MCMC_MAX_FREE:
        raise ValueError("1..%d free parameters" % MCMC_MAX_FREE)
    spec.n_free = len(targets)
    for k, (kind, index, pos) in enumerate(targets):
        p = spec.param[k]
        p.kind, p.index, p.pos, p.lo, p.hi = int(kind), int(index), int(pos), float(lo[k]), float(hi[k])
    return spec


def make_mcmc(n_walkers, targets, lo, hi, n_sc, n_obs_series, sc_per_member=False, thin=1, seed=0, stretch=2.0):
    """SimplypMcmc for ``targets`` [(kind, index, pos)] (``MCMC_MEMBER`` / ``MCMC_SC_ALL`` / ``MCMC_SC_AT``) with the
    prior box ``[lo[k], hi[k]]``."""
    mc = _free_params(SimplypMcmc(), targets, lo, hi)
    mc.n_walkers, mc.n_sc, mc.n_obs_series = int(n_walkers), int(n_sc), int(n_obs_series)
    mc.sc_per_member, mc.thin = 1 if sc_per_member else 0, int(thin)
    mc.seed, mc.stretch = _u64(seed), float(stretch)
    return mc


def make_mcmc_state(walkers, lp, proposals, log_z, out_of_box, iteration, accepted, chain, chain_lp, n_saved,
                    chain_base=0):
    """SimplypMcmcState from device pointers (torch ``.data_ptr()`` integers)."""
    st = SimplypMcmcState()
    st.walkers, st.lp, st.proposals, st.log_z = walkers, lp, proposals, log_z
    st.out_of_box, st.iteration, st.accepted = out_of_box, iteration, accepted
    st.chain, st.chain_lp, st.n_saved, st.chain_base = chain, chain_lp, int(n_saved), int(chain_base)
    return st


def mcmc_propose_device(mc, state, half, member_ptr, sc_ptr, stream_ptr):
    """Proposals of walker half ``half`` into its member (and SC) rows; asynchronous on ``stream_ptr``."""
    lib = require_device()
    _check(lib.simplyp_mcmc_propose_device(C.byref(mc), C.byref(state), int(half), member_ptr, sc_ptr, stream_ptr))


def mcmc_accept_device(mc, state, half, stats_ptr, diag_ptr, stream_ptr):
    """Metropolis-Hastings step of half ``half`` from its calibration statistics; asynchronous on ``stream_ptr``."""
    lib = require_device()
    _check(lib.simplyp_mcmc_accept_device(C.byref(mc), C.byref(state), int(half), stats_ptr, diag_ptr, stream_ptr))


def mcmc_init_device(mc, state, stats_ptr, diag_ptr, stream_ptr):
    """lp of the current walkers from the statistics of one run of all W rows; asynchronous on ``stream_ptr``."""
    lib = require_device()
    _check(lib.simplyp_mcmc_init_device(C.byref(mc), C.byref(state), stats_ptr, diag_ptr, stream_ptr))


def predictive_draws_device(dims, out_ptr, member_ptr, sc_ptr, diag_ptr, series_desc_ptr, n_series, draws_ptr,
                            n_members_total, member_offset, obs_error, seed, stream_ptr):
    """Draws of the simulated series of one full-output chunk into its columns of draws [V][D][M_total];
    asynchronous on ``stream_ptr``."""
    lib = require_device()
    _check(lib.simplyp_predictive_draws_device(C.byref(dims), out_ptr, member_ptr, sc_ptr, diag_ptr, series_desc_ptr,
                                               int(n_series), draws_ptr, int(n_members_total), int(member_offset),
                                               1 if obs_error else 0, _u64(seed), stream_ptr))


def period_aggregates_device(dims, out_ptr, member_ptr, sc_ptr, diag_ptr, series_desc, period_bounds, wb_reaches,
                             values_ptr, n_members_total, member_offset, stream_ptr):
    """Period aggregates of one full-output chunk into its columns of values [V P][M_total]; ``series_desc`` [V][3],
    ``period_bounds`` [P][2] and ``wb_reaches`` [n] are host int32 arrays, passed to the kernel by value.
    Asynchronous on ``stream_ptr``."""
    lib = require_device()
    desc = np.ascontiguousarray(series_desc, dtype=np.int32).reshape(-1, 3)
    bounds = np.ascontiguousarray(period_bounds, dtype=np.int32).reshape(-1, 2)
    wb = np.ascontiguousarray(wb_reaches, dtype=np.int32).reshape(-1)
    ip = C.POINTER(C.c_int32)
    _check(lib.simplyp_period_aggregates_device(C.byref(dims), out_ptr, member_ptr, sc_ptr, diag_ptr,
                                                desc.ctypes.data_as(ip), desc.shape[0], bounds.ctypes.data_as(ip),
                                                bounds.shape[0], wb.ctypes.data_as(ip) if wb.size else None, wb.size,
                                                values_ptr, int(n_members_total), int(member_offset), stream_ptr))


def nanquantile_workspace_bytes(n_rows, n_cols):
    n = load().simplyp_nanquantile_workspace_bytes(int(n_rows), int(n_cols))
    if n < 0:
        _check(int(n))
    return int(n)


def nanquantile_device(x_ptr, n_rows, n_cols, q, quant_ptr, mean_ptr, count_ptr, ws_ptr, ws_bytes, stream_ptr):
    """np.nanquantile of every row of x [n_rows][n_cols] (``q`` a host sequence) into quantiles [n_q][n_rows], the
    mean and the count of the non-NaN entries; asynchronous on ``stream_ptr``."""
    lib = require_device()
    qa = (C.c_double * max(len(q), 1))(*[float(v) for v in q])
    _check(lib.simplyp_nanquantile_device(x_ptr, int(n_rows), int(n_cols), qa, len(q), quant_ptr, mean_ptr, count_ptr,
                                          ws_ptr, int(ws_bytes), stream_ptr))


def make_sobol(targets, lo, hi, n_sc, n_base, skip=0, sc_per_member=False, second_order=False):
    """SimplypSobol for ``targets`` [(kind, index, pos)] (as :func:`make_mcmc`) with the boxes ``[lo[k], hi[k]]``."""
    sb = _free_params(SimplypSobol(), targets, lo, hi)
    sb.n_sc = int(n_sc)
    sb.sc_per_member, sb.second_order = 1 if sc_per_member else 0, 1 if second_order else 0
    sb.n_base, sb.skip = int(n_base), int(skip)
    return sb


def sobol_design_device(sb, member_offset, n_members, member_ptr, sc_ptr, stream_ptr):
    """Target columns of design members [member_offset, member_offset + n_members); asynchronous on ``stream_ptr``."""
    lib = require_device()
    _check(lib.simplyp_sobol_design_device(C.byref(sb), int(member_offset), int(n_members), member_ptr, sc_ptr,
                                           stream_ptr))


def sobol_outputs_device(stats_ptr, diag_ptr, n_members, n_obs_series, n_sc, rows_ptr, n_rows, y_ptr, stream_ptr):
    """Objective rows Y [n_rows][M] from the fused statistics; asynchronous on ``stream_ptr``."""
    lib = require_device()
    _check(lib.simplyp_sobol_outputs_device(stats_ptr, diag_ptr, int(n_members), int(n_obs_series), int(n_sc),
                                            rows_ptr, int(n_rows), y_ptr, stream_ptr))


def sobol_workspace_bytes(sb, n_rows):
    n = load().simplyp_sobol_workspace_bytes(C.byref(sb), int(n_rows))
    if n < 0:
        _check(int(n))
    return int(n)


def sobol_indices_device(sb, y_ptr, n_rows, n_boot, conf_z, seed, S1, ST, S1_conf, ST_conf, S2, S2_conf, mean, var,
                         n_used, ws_ptr, ws_bytes, stream_ptr):
    """Sobol' indices and bootstrap confidences of every row of Y [n_rows][N P]; asynchronous on ``stream_ptr``."""
    lib = require_device()
    _check(lib.simplyp_sobol_indices_device(C.byref(sb), y_ptr, int(n_rows), int(n_boot), float(conf_z),
                                            _u64(seed), S1, ST, S1_conf, ST_conf, S2, S2_conf,
                                            mean, var, n_used, ws_ptr, int(ws_bytes), stream_ptr))


def make_morris(targets, lo, hi, n_sc, n_trajectories, num_levels=4, n_candidates=0, sc_per_member=False, seed=0):
    """SimplypMorris for ``targets`` [(kind, index, pos)] (as :func:`make_mcmc`) with the boxes ``[lo[k], hi[k]]``;
    ``n_candidates`` 0 takes trajectory i from candidate i."""
    mo = _free_params(SimplypMorris(), targets, lo, hi)
    mo.n_sc, mo.sc_per_member, mo.num_levels = int(n_sc), 1 if sc_per_member else 0, int(num_levels)
    mo.n_trajectories, mo.n_candidates, mo.seed = int(n_trajectories), int(n_candidates or 0), _u64(seed)
    return mo


def morris_workspace_bytes(mo, n_rows):
    n = load().simplyp_morris_workspace_bytes(C.byref(mo), int(n_rows))
    if n < 0:
        _check(int(n))
    return int(n)


def morris_select_device(mo, selected_ptr, ws_ptr, ws_bytes, stream_ptr):
    """Indices selected [r] int32 of the optimised trajectories; asynchronous on ``stream_ptr``."""
    _check(require_device().simplyp_morris_select_device(C.byref(mo), selected_ptr, ws_ptr, int(ws_bytes), stream_ptr))


def morris_design_device(mo, selected_ptr, member_offset, n_members, member_ptr, sc_ptr, stream_ptr):
    """Target columns of design members [member_offset, member_offset + n_members); asynchronous on ``stream_ptr``."""
    _check(require_device().simplyp_morris_design_device(C.byref(mo), selected_ptr, int(member_offset), int(n_members),
                                                         member_ptr, sc_ptr, stream_ptr))


def morris_effects_device(mo, selected_ptr, y_ptr, n_rows, n_boot, conf_z, mu, mu_star, sigma, mu_star_conf, n_used,
                          ws_ptr, ws_bytes, stream_ptr):
    """Elementary-effect statistics of every row of Y [n_rows][r (K + 1)]; asynchronous on ``stream_ptr``."""
    _check(require_device().simplyp_morris_effects_device(C.byref(mo), selected_ptr, y_ptr, int(n_rows), int(n_boot),
                                                          float(conf_z), mu, mu_star, sigma, mu_star_conf, n_used,
                                                          ws_ptr, int(ws_bytes), stream_ptr))


def make_de(n_population, targets, lo, hi, n_sc, n_rows, sc_per_member=False, strategy="best1bin",
            mutation=(0.5, 1.0), recombination=0.7, tol=0.01, tol_abs=0.0, seed=0):
    """SimplypDe for ``targets`` [(kind, index, pos)] (as :func:`make_mcmc`) with the boxes ``[lo[k], hi[k]]``."""
    de = _free_params(SimplypDe(), targets, lo, hi)
    de.n_population, de.n_sc, de.n_rows = int(n_population), int(n_sc), int(n_rows)
    de.sc_per_member, de.strategy = 1 if sc_per_member else 0, DE_STRATEGIES[strategy]
    de.seed = _u64(seed)
    de.mutation_lo, de.mutation_hi = float(mutation[0]), float(mutation[1])
    de.recombination, de.tol, de.tol_abs = float(recombination), float(tol), float(tol_abs)
    return de


def make_de_state(population, energy, trial, flags, weights, generation, best, converged, converged_at, n_failed,
                  history, n_history, history_base=0):
    """SimplypDeState from device pointers (torch ``.data_ptr()`` integers)."""
    st = SimplypDeState()
    st.population, st.energy, st.trial, st.flags, st.weights = population, energy, trial, flags, weights
    st.generation, st.best, st.converged, st.converged_at = generation, best, converged, converged_at
    st.n_failed, st.history, st.n_history, st.history_base = n_failed, history, int(n_history), int(history_base)
    return st


def de_trial_device(de, state, member_ptr, sc_ptr, stream_ptr):
    """Trials of every member into ``trial`` and the target columns of its rows; asynchronous on ``stream_ptr``."""
    _check(require_device().simplyp_de_trial_device(C.byref(de), C.byref(state), member_ptr, sc_ptr, stream_ptr))


def de_select_device(de, state, y_ptr, diag_ptr, stream_ptr):
    """Selection, reduction and history row of one generation from the trials' objective rows y [R][N] and diag;
    asynchronous on ``stream_ptr``."""
    _check(require_device().simplyp_de_select_device(C.byref(de), C.byref(state), y_ptr, diag_ptr, stream_ptr))


def de_init_device(de, state, y_ptr, diag_ptr, stream_ptr):
    """Energies, best member and history row 0 from the population's objective rows y [R][N] and diag; asynchronous
    on ``stream_ptr``."""
    _check(require_device().simplyp_de_init_device(C.byref(de), C.byref(state), y_ptr, diag_ptr, stream_ptr))


def de_scale_device(de, unit_ptr, n, out_ptr, stream_ptr):
    """Parameter values out [n][K] of unit-cube rows unit [n][K]; asynchronous on ``stream_ptr``."""
    _check(require_device().simplyp_de_scale_device(C.byref(de), unit_ptr, int(n), out_ptr, stream_ptr))


def make_nsga2(n_population, targets, lo, hi, n_sc, sense, sc_per_member=False, crossover=0.9, mutation=None,
               eta_c=15.0, eta_m=20.0, seed=0):
    """SimplypNsga2 for ``targets`` [(kind, index, pos)] (as :func:`make_mcmc`) with the boxes ``[lo[k], hi[k]]`` and
    the objective senses ``sense`` [M] (+1 maximised, -1 minimised); ``mutation`` None is 1/K."""
    ns = _free_params(SimplypNsga2(), targets, lo, hi)
    ns.n_population, ns.n_sc, ns.n_objectives = int(n_population), int(n_sc), len(sense)
    ns.sc_per_member = 1 if sc_per_member else 0
    for m, v in enumerate(sense):
        ns.sense[m] = float(v)
    ns.seed = _u64(seed)
    ns.crossover = float(crossover)
    ns.mutation = 1.0 / ns.n_free if mutation is None else float(mutation)
    ns.eta_c, ns.eta_m = float(eta_c), float(eta_m)
    return ns


def make_nsga2_state(population, objectives, rank, crowding, offspring, generation, n_failed, history, n_history,
                     workspace, workspace_bytes, history_base=0):
    """SimplypNsga2State from device pointers (torch ``.data_ptr()`` integers)."""
    st = SimplypNsga2State()
    st.population, st.objectives, st.rank, st.crowding = population, objectives, rank, crowding
    st.offspring, st.generation, st.n_failed = offspring, generation, n_failed
    st.history, st.n_history, st.history_base = history, int(n_history), int(history_base)
    st.workspace, st.workspace_bytes = workspace, int(workspace_bytes)
    return st


def nsga2_workspace_bytes(ns):
    n = load().simplyp_nsga2_workspace_bytes(C.byref(ns))
    if n < 0:
        _check(int(n))
    return int(n)


def nsga2_init_device(ns, state, y_ptr, diag_ptr, stream_ptr):
    """Objectives, ranks, crowding and history row 0 of the population from its objective rows y [M][N] and diag;
    asynchronous on ``stream_ptr``."""
    _check(require_device().simplyp_nsga2_init_device(C.byref(ns), C.byref(state), y_ptr, diag_ptr, stream_ptr))


def nsga2_offspring_device(ns, state, member_ptr, sc_ptr, stream_ptr):
    """Offspring of every pair into ``offspring`` and the target columns of their rows; asynchronous on
    ``stream_ptr``."""
    _check(require_device().simplyp_nsga2_offspring_device(C.byref(ns), C.byref(state), member_ptr, sc_ptr,
                                                           stream_ptr))


def nsga2_survive_device(ns, state, y_ptr, diag_ptr, stream_ptr):
    """Ranking, crowding, survival and history row of one generation from the offspring's objective rows y [M][N] and
    diag; asynchronous on ``stream_ptr``."""
    _check(require_device().simplyp_nsga2_survive_device(C.byref(ns), C.byref(state), y_ptr, diag_ptr, stream_ptr))


def workspace_bytes(dims, calibrate, rank_stats=False):
    n = load().simplyp_workspace_bytes(C.byref(dims), (1 if calibrate else 0) | (2 if (calibrate and rank_stats) else 0))
    if n < 0:
        _check(int(n))
    return int(n)


def launch_count():
    return int(load().simplyp_launch_count())


def measure_fp64_latency(device=0):
    require_device()
    return float(load().simplyp_measure_fp64_latency(device))


def measure_fp64_peak(device=0, repeats=3):
    require_device()
    return float(load().simplyp_measure_fp64_peak(device, repeats))
