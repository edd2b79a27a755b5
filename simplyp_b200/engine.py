"""Device-resident execution of the integrator: torch owns memory and streams, the C-ABI does the work.

``Engine`` keeps forcing / parameters / observations resident in HBM as torch tensors and calls the
``*_device`` entry points of ``libsimplyp_b200.so`` with raw pointers on torch's current stream.
PyTorch is plumbing only (allocation, streams, ``torch.distributed``); every arithmetic step of the
path runs in the hand-written kernels.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _cabi
from . import packing as pk


def _torch():
    import torch
    return torch


def half_free_bytes(eng):
    """Half of the free memory of ``eng``'s device: the most the buffers of an ensemble driver may take, and the default
    workspace budget of :meth:`Engine.calibrate`.  A driver that captures CUDA graphs takes its budget up front, so
    that nothing queries memory during a capture."""
    return eng.free_bytes() // 2


def check_device_memory(eng, nbytes, what, hint):
    """``ValueError`` "<what> <GB>, more than half of the free device memory: <hint>" if ``nbytes`` exceed
    :func:`half_free_bytes`; asks ``eng`` for nothing but ``free_bytes()``, so a driver calls it before any device
    work."""
    if nbytes > half_free_bytes(eng):
        raise ValueError("%s %.1f GB, more than half of the free device memory: %s" % (what, nbytes / 1e9, hint))


class Engine:
    """One engine per process / GPU."""

    def __init__(self, device=None):
        torch = _torch()
        _cabi.require_device()
        if not torch.cuda.is_available():
            raise _cabi.SimplypError("torch sees no CUDA device: simplyp_b200 has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        self._ws = None

    # ------------------------------------------------------------------ helpers
    def to_device(self, a, dtype=None):
        torch = _torch()
        if isinstance(a, torch.Tensor):
            return a.to(self.device).contiguous()
        a = np.ascontiguousarray(a, dtype=dtype)
        return torch.from_numpy(a).to(self.device)

    def _workspace(self, nbytes):
        torch = _torch()
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = None
            self._ws = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.device)
        return self._ws

    def free_bytes(self):
        torch = _torch()
        free, _total = torch.cuda.mem_get_info(self.device)
        return int(free)

    def context(self):
        """This engine's device as torch's current device."""
        return _torch().cuda.device(self.device)

    def _call(self, fn, *args):
        """``fn(*args, stream)`` on this device, ``stream`` being torch's current stream."""
        with self.context():
            fn(*args, _torch().cuda.current_stream().cuda_stream)

    def capture(self, step):
        """``step()``, which only enqueues work, captured into a CUDA graph on this device."""
        torch = _torch()
        g = torch.cuda.CUDAGraph()
        with self.context(), torch.cuda.graph(g):
            step()
        return g

    @staticmethod
    def _sc_sets(sc_params):
        """SC parameters as [Msc][S][NP_SC]: a [S][NP_SC] matrix is the one set of every member."""
        return sc_params.unsqueeze(0) if sc_params.dim() == 2 else sc_params

    @classmethod
    def _shapes(cls, forcing, member_params, sc_params):
        D = forcing.shape[0]
        M = member_params.shape[0]
        sc_params = cls._sc_sets(sc_params)
        Msc, S = sc_params.shape[0], sc_params.shape[1]
        assert forcing.shape[1] == pk.NF and member_params.shape[1] == pk.NP_MEMBER and sc_params.shape[2] == pk.NP_SC
        return D, M, Msc, S, sc_params

    @classmethod
    def _output_dims(cls, out, sc_params):
        """(SimplypDims, SC parameter sets) of a full-output chunk ``out`` [M][S][D][25]."""
        sc_params = cls._sc_sets(sc_params)
        return _cabi.make_dims(out.shape[0], out.shape[1], out.shape[2], sc_params.shape[0], 0, 0), sc_params

    # ------------------------------------------------------------------ full output
    def run(self, forcing, member_params, sc_params, parent_offsets, parent_ids, opt, out=None, diag=None):
        """All tensors on this device, fp64.  Returns (out [M][S][D][25], diag [M][S][4] int64); asynchronous."""
        torch = _torch()
        D, M, Msc, S, sc_params = self._shapes(forcing, member_params, sc_params)
        n_edges = int(parent_offsets[-1])
        dims = _cabi.make_dims(M, S, D, Msc, 0, n_edges)
        if out is None:
            out = torch.empty((M, S, D, pk.NOUT), dtype=torch.float64, device=self.device)
        if diag is None:
            diag = torch.zeros((M, S, pk.NDIAG), dtype=torch.int64, device=self.device)
        ws = self._workspace(_cabi.workspace_bytes(dims, False))
        self._call(_cabi.run_device, dims, opt, forcing.data_ptr(), member_params.data_ptr(), sc_params.data_ptr(),
                   parent_offsets, parent_ids, out.data_ptr(), diag.data_ptr(), ws.data_ptr())
        return out, diag

    # ------------------------------------------------------------------ fused statistics
    def calibrate(self, forcing, member_params, sc_params, parent_offsets, parent_ids, obs, obs_desc, opt,
                  stats=None, diag=None, max_workspace_bytes=None, peer_gather=None, phi=None, phi_col=None):
        """Returns (stats [M][V][10], diag [M][S][4]); asynchronous on the current stream.

        With ``phi`` (a contiguous [M][P] fp64 device tensor) and ``phi_col`` ([V] ints) the log-likelihood of series v
        has the AR(1) error model with phi = ``phi[m][phi_col[v]]`` (``simplyp_calibrate_ar1_device``); series with
        ``phi_col[v] < 0`` keep the iid value.

        With ``peer_gather`` (an :class:`ensemble.PeerGather`; the members given here are this rank's shard) the
        statistics of ALL ranks come back, [M_total][V][10]: the kernel stores them into every rank's buffer and a flag
        exchange ends the call on the stream — no collective follows.

        The workspace grows with the members: M*S*D*32 bytes of flux exchange for networks (S > 1) and M*V*D*8
        bytes of simulated values with ``opt.rank_stats`` or ``phi``; members are processed in chunks that keep it under
        ``max_workspace_bytes`` (default: half of the free HBM).
        """
        torch = _torch()
        D, M, Msc, S, sc_params = self._shapes(forcing, member_params, sc_params)
        V = obs.shape[0]
        n_edges = int(parent_offsets[-1])
        if phi is not None and (phi.dim() != 2 or phi.shape[0] != M or phi.dtype != torch.float64
                                or not phi.is_contiguous() or phi_col is None or len(phi_col) != V):
            raise ValueError("phi must be a contiguous [M][P] float64 tensor and phi_col hold one column per series")
        if stats is None and peer_gather is None:
            stats = torch.empty((M, V, pk.NSTAT), dtype=torch.float64, device=self.device)
        if diag is None:
            diag = torch.zeros((M, S, pk.NDIAG), dtype=torch.int64, device=self.device)
        chunk = M
        keep_sim = bool(opt.rank_stats) or phi is not None
        per_member = (32 * S * D if S > 1 else 0) + (8 * V * D if keep_sim else 0)
        if per_member > 0:
            budget = max_workspace_bytes if max_workspace_bytes is not None else half_free_bytes(self)
            chunk = max(1, min(M, int(budget // per_member)))
        if peer_gather is not None:
            if chunk < M or keep_sim or M != peer_gather.hi - peer_gather.lo:
                raise _cabi.SimplypError("peer_gather: one launch of this rank's whole shard, without rank statistics "
                                         "or an AR(1) error model")
            dims = _cabi.make_dims(M, S, D, 1 if Msc == 1 else M, V, n_edges)
            ws = self._workspace(_cabi.workspace_bytes(dims, True, False))
            desc, gathered = peer_gather.descriptor()
            self._call(_cabi.calibrate_gather_device, dims, opt, forcing.data_ptr(), member_params.data_ptr(),
                       sc_params.data_ptr(), parent_offsets, parent_ids, obs.data_ptr(), obs_desc.data_ptr(), desc,
                       diag.data_ptr(), ws.data_ptr())
            return gathered, diag
        for m0 in range(0, M, chunk):
            m1 = min(M, m0 + chunk)
            dims = _cabi.make_dims(m1 - m0, S, D, 1 if Msc == 1 else (m1 - m0), V, n_edges)
            ws = self._workspace(_cabi.workspace_bytes(dims, True, keep_sim))
            scp = sc_params if Msc == 1 else sc_params[m0:m1]
            args = (dims, opt, forcing.data_ptr(), member_params[m0:m1].data_ptr(), scp.data_ptr(), parent_offsets,
                    parent_ids, obs.data_ptr(), obs_desc.data_ptr())
            tail = (stats[m0:m1].data_ptr(), diag[m0:m1].data_ptr(), ws.data_ptr())
            if phi is None:
                self._call(_cabi.calibrate_device, *args, *tail)
            else:
                ar1 = _cabi.make_ar1(phi[m0:m1].data_ptr(), phi.shape[1], phi_col)
                self._call(_cabi.calibrate_ar1_device, *args, ar1, *tail)
        return stats, diag

    # ------------------------------------------------------------------ receiving water body
    WATERBODY_COLUMNS = ["Q_cumecs", "Msus_kg/day", "TDP_kg/day", "PP_kg/day", "SS_mgl", "TDP_mgl", "PP_mgl",
                         "TP_mgl", "TP_kg/day", "SRP_mgl", "SRP_kg/day"]

    def sum_to_waterbody(self, out, member_params, sc_params, reaches):
        """Reference ``sum_to_waterbody`` (``model.py:851-900``) for every member of a full-output run, on the
        device: ``out`` [M][S][D][25] from :meth:`run`, ``reaches`` = run-order indices of the reaches flagged
        ``In_final_flux? == 1``.  Returns [M][D][11] (columns ``WATERBODY_COLUMNS``); asynchronous."""
        torch = _torch()
        dims, sc_params = self._output_dims(out, sc_params)
        r = torch.as_tensor(np.asarray(reaches, dtype=np.int32), device=self.device)
        wb = torch.empty((out.shape[0], out.shape[2], len(self.WATERBODY_COLUMNS)), dtype=torch.float64,
                         device=self.device)
        self._call(_cabi.sum_to_waterbody_device, dims, out.data_ptr(), sc_params.data_ptr(), member_params.data_ptr(),
                   r.data_ptr(), int(r.numel()), wb.data_ptr())
        return wb

    # ------------------------------------------------------------------ posterior predictive bands
    def predictive_draws(self, out, member_params, sc_params, diag, series_desc, draws, member_offset=0,
                         obs_error=False, seed=0):
        """Simulated series of a full-output chunk (``out`` [Mc][S][D][25], ``diag`` [Mc][S][4] from :meth:`run`)
        written into columns ``member_offset .. member_offset + Mc`` of ``draws`` [V][D][M_total] for the series
        ``series_desc`` [V][2] int32 (run-order reach, ``packing.VAR_KINDS`` index), optionally through the
        likelihood's error model (``simplyp_predictive_draws_device``).  Returns ``draws``; asynchronous."""
        dims, sc_params = self._output_dims(out, sc_params)
        self._call(_cabi.predictive_draws_device, dims, out.data_ptr(), member_params.data_ptr(), sc_params.data_ptr(),
                   diag.data_ptr(), series_desc.data_ptr(), series_desc.shape[0], draws.data_ptr(), draws.shape[2],
                   member_offset, obs_error, seed)
        return draws

    def period_aggregates(self, out, member_params, sc_params, diag, series_desc, period_bounds, wb_reaches, values,
                          member_offset=0):
        """Period means, loads and flow-weighted concentrations of a full-output chunk (``out`` [Mc][S][D][25],
        ``diag`` [Mc][S][4] from :meth:`run`) written into columns ``member_offset .. member_offset + Mc`` of
        ``values`` [V P][M_total], row v P + p (``simplyp_period_aggregates_device``).  ``series_desc`` [V][3] =
        (run-order reach or ``_cabi.PERIOD_WATERBODY``, ``packing.VAR_KINDS`` index, ``_cabi.PERIOD_STATS`` code),
        ``period_bounds`` [P][2] (first and last day) and ``wb_reaches`` (run-order reaches of the water body) are
        host arrays.  Returns ``values``; asynchronous."""
        dims, sc_params = self._output_dims(out, sc_params)
        self._call(_cabi.period_aggregates_device, dims, out.data_ptr(), member_params.data_ptr(), sc_params.data_ptr(),
                   diag.data_ptr(), series_desc, period_bounds, wb_reaches, values.data_ptr(), values.shape[1],
                   member_offset)
        return values

    def nanquantile(self, x, q, quantiles=None, mean=None, count=None):
        """``np.nanquantile(x, q, axis=-1)`` of a [R][N] fp64 matrix, bitwise, with the mean and the count of the
        non-NaN entries of every row (``simplyp_nanquantile_device``).  Returns (quantiles [n_q][R], mean [R],
        count [R] int64); asynchronous.  Rows longer than shared memory holds use this engine's workspace."""
        torch = _torch()
        if x.dim() != 2 or x.dtype != torch.float64 or not x.is_contiguous():
            raise ValueError("nanquantile takes a contiguous [R][N] float64 matrix")
        R, N = x.shape
        if quantiles is None:
            quantiles = torch.empty((len(q), R), dtype=torch.float64, device=self.device)
        if mean is None:
            mean = torch.empty(R, dtype=torch.float64, device=self.device)
        if count is None:
            count = torch.empty(R, dtype=torch.int64, device=self.device)
        need = _cabi.nanquantile_workspace_bytes(R, N)
        ws = self._workspace(need) if need > 0 else None
        self._call(_cabi.nanquantile_device, x.data_ptr(), R, N, q, quantiles.data_ptr(), mean.data_ptr(),
                   count.data_ptr(), ws.data_ptr() if ws is not None else None, need)
        return quantiles, mean, count

    # ------------------------------------------------------------------ Sobol' sensitivity
    def sobol_design(self, sb, member_params, sc_params, member_offset=0, n_members=None):
        """Write the target columns of design members ``member_offset .. member_offset + n_members`` (default: to
        the end) of ``member_params`` [N P][NP_MEMBER] and ``sc_params`` ([N P] or [1])[S][NP_SC] for the
        :class:`_cabi.SimplypSobol` ``sb`` (``simplyp_sobol_design_device``).  Asynchronous."""
        if n_members is None:
            n_members = member_params.shape[0] - member_offset
        self._call(_cabi.sobol_design_device, sb, member_offset, n_members, member_params.data_ptr(),
                   sc_params.data_ptr())
        return member_params, sc_params

    def sobol_outputs(self, stats, diag, rows, y):
        """Objective rows ``y`` [R][M] from the fused statistics ``stats`` [M][V][10] and ``diag`` [M][S][4];
        ``rows`` [R][2] int32 on the device = (series, ``packing.STAT_NAMES`` slot, or -1 for the sampler's lp)
        (``simplyp_sobol_outputs_device``).  Asynchronous."""
        self._call(_cabi.sobol_outputs_device, stats.data_ptr(), diag.data_ptr(), stats.shape[0], stats.shape[1],
                   diag.shape[1], rows.data_ptr(), rows.shape[0], y.data_ptr())
        return y

    def sobol_indices(self, sb, y, n_boot, conf_z, seed, out=None):
        """Sobol' indices of every row of ``y`` [R][N P] with bootstrap confidences (``simplyp_sobol_indices_device``).
        Returns a dict of device tensors S1, ST, S1_conf, ST_conf [R][K], S2, S2_conf [R][K][K] (second order
        only), mean, var [R] and n_used [R]; ``out`` may give them preallocated.  Asynchronous."""
        torch = _torch()
        if y.dim() != 2 or y.dtype != torch.float64 or not y.is_contiguous():
            raise ValueError("sobol_indices takes a contiguous [R][N P] float64 matrix")
        R, K = y.shape[0], sb.n_free
        f64 = dict(dtype=torch.float64, device=self.device)
        if out is None:
            out = {k: torch.empty((R, K), **f64) for k in ("S1", "ST", "S1_conf", "ST_conf")}
            if sb.second_order:
                out.update({k: torch.empty((R, K, K), **f64) for k in ("S2", "S2_conf")})
            out.update(mean=torch.empty(R, **f64), var=torch.empty(R, **f64),
                       n_used=torch.empty(R, dtype=torch.int64, device=self.device))
        need = _cabi.sobol_workspace_bytes(sb, R)
        ws = self._workspace(need)

        def ptr(k):
            return out[k].data_ptr() if k in out else None
        self._call(_cabi.sobol_indices_device, sb, y.data_ptr(), R, n_boot, conf_z, seed, ptr("S1"), ptr("ST"),
                   ptr("S1_conf"), ptr("ST_conf"), ptr("S2"), ptr("S2_conf"), ptr("mean"), ptr("var"), ptr("n_used"),
                   ws.data_ptr(), need)
        return out

    # ------------------------------------------------------------------ Morris screening
    def morris_select(self, mo, selected=None):
        """Indices [r] int32 (device) of the trajectories the greedy spread search picks among the
        :class:`_cabi.SimplypMorris` ``mo``'s candidates (``simplyp_morris_select_device``).  Asynchronous."""
        torch = _torch()
        if selected is None:
            selected = torch.empty(mo.n_trajectories, dtype=torch.int32, device=self.device)
        need = _cabi.morris_workspace_bytes(mo, 0)
        ws = self._workspace(need)
        self._call(_cabi.morris_select_device, mo, selected.data_ptr(), ws.data_ptr(), need)
        return selected

    def morris_design(self, mo, member_params, sc_params, selected=None, member_offset=0, n_members=None):
        """Write the target columns of design members ``member_offset .. member_offset + n_members`` (default: to the
        end) of ``member_params`` [r (K+1)][NP_MEMBER] and ``sc_params`` ([r (K+1)] or [1])[S][NP_SC]; ``selected``
        (from :meth:`morris_select`) is needed when ``mo`` has candidates (``simplyp_morris_design_device``).
        Asynchronous."""
        if n_members is None:
            n_members = member_params.shape[0] - member_offset
        self._call(_cabi.morris_design_device, mo, selected.data_ptr() if selected is not None else None,
                   member_offset, n_members, member_params.data_ptr(), sc_params.data_ptr())
        return member_params, sc_params

    def morris_effects(self, mo, y, n_boot, conf_z, selected=None, out=None):
        """Elementary-effect statistics of every row of ``y`` [R][r (K+1)] (``simplyp_morris_effects_device``).
        Returns a dict of device tensors mu, mu_star, sigma, mu_star_conf [R][K] and n_used [R]; ``out`` may give them
        preallocated.  Asynchronous."""
        torch = _torch()
        if y.dim() != 2 or y.dtype != torch.float64 or not y.is_contiguous():
            raise ValueError("morris_effects takes a contiguous [R][r (K + 1)] float64 matrix")
        R, K = y.shape[0], mo.n_free
        if out is None:
            out = {k: torch.empty((R, K), dtype=torch.float64, device=self.device)
                   for k in ("mu", "mu_star", "sigma", "mu_star_conf")}
            out["n_used"] = torch.empty(R, dtype=torch.int64, device=self.device)
        need = _cabi.morris_workspace_bytes(mo, R)
        ws = self._workspace(need)
        self._call(_cabi.morris_effects_device, mo, selected.data_ptr() if selected is not None else None,
                   y.data_ptr(), R, n_boot, conf_z, out["mu"].data_ptr(), out["mu_star"].data_ptr(),
                   out["sigma"].data_ptr(), out["mu_star_conf"].data_ptr(), out["n_used"].data_ptr(), ws.data_ptr(),
                   need)
        return out

    # ------------------------------------------------------------------ differential evolution
    def de_trial(self, de, state, member_params, sc_params):
        """Trials of the :class:`_cabi.SimplypDe` population ``state`` into its trial buffer and the target columns of
        ``member_params`` [N][NP_MEMBER] / ``sc_params`` ([N] or [1])[S][NP_SC] (``simplyp_de_trial_device``).
        Asynchronous."""
        self._call(_cabi.de_trial_device, de, state, member_params.data_ptr(), sc_params.data_ptr())

    def de_select(self, de, state, y, diag):
        """Selection of one generation from the trials' objective rows ``y`` [R][N] (:meth:`sobol_outputs`) and
        ``diag`` [N][S][4] (``simplyp_de_select_device``).  Asynchronous."""
        self._call(_cabi.de_select_device, de, state, y.data_ptr(), diag.data_ptr())

    def de_scale(self, de, unit, out):
        """Parameter values ``out`` [n][K] of unit-cube rows ``unit`` [n][K] (``simplyp_de_scale_device``).
        Asynchronous."""
        self._call(_cabi.de_scale_device, de, unit.data_ptr(), unit.shape[0], out.data_ptr())

    def de_init(self, de, state, y, diag):
        """Energies, best member and history row 0 from the population's objective rows ``y`` [R][N] and ``diag``
        (``simplyp_de_init_device``).  Asynchronous."""
        self._call(_cabi.de_init_device, de, state, y.data_ptr(), diag.data_ptr())

    # ------------------------------------------------------------------ NSGA-II
    def nsga2_init(self, ns, state, y, diag):
        """Objectives, ranks, crowding and history row 0 of the population from its objective rows ``y`` [M][N] and
        ``diag`` [N][S][4] (``simplyp_nsga2_init_device``).  Asynchronous."""
        self._call(_cabi.nsga2_init_device, ns, state, y.data_ptr(), diag.data_ptr())

    def nsga2_offspring(self, ns, state, member_params, sc_params):
        """Enqueue the offspring of one NSGA-II generation into ``state.offspring`` and the target columns of
        ``member_params`` [N][NP_MEMBER] / ``sc_params`` ([N] or [1])[S][NP_SC] (``simplyp_nsga2_offspring_device``)."""
        self._call(_cabi.nsga2_offspring_device, ns, state, member_params.data_ptr(), sc_params.data_ptr())

    def nsga2_survive(self, ns, state, y, diag):
        """Enqueue the survival of one NSGA-II generation from the offspring's objective rows ``y`` [M][N] and ``diag``
        [N][S][4] (``simplyp_nsga2_survive_device``).  Asynchronous."""
        self._call(_cabi.nsga2_survive_device, ns, state, y.data_ptr(), diag.data_ptr())

    # ------------------------------------------------------------------ Thornthwaite PET
    def thornthwaite_pet(self, t_air, month_start, year_is_leap, latitude_deg, out=None, out_stride=1):
        """Reference ``daily_PET`` (``inputs.py:232-312``) on the device: ``t_air`` [D] (device or host),
        ``month_start`` [n_months + 1] day index at which each calendar month of the record starts,
        ``year_is_leap`` [n_months / 12]; returns PET [D] in mm/day (or writes ``out`` with ``out_stride``,
        e.g. column 1 of a forcing matrix: ``out=forcing[:, 1], out_stride=4``); asynchronous."""
        torch = _torch()
        t = self.to_device(t_air, np.float64)
        ms = torch.as_tensor(np.asarray(month_start, dtype=np.int32), device=self.device)
        lp = torch.as_tensor(np.asarray(year_is_leap, dtype=np.int32), device=self.device)
        D, NM = int(t.numel()), int(ms.numel()) - 1
        if out is None:
            out = torch.empty(D, dtype=torch.float64, device=self.device)
            out_stride = 1
        self._call(_cabi.thornthwaite_pet_device, D, NM, t.data_ptr(), 1, ms.data_ptr(), lp.data_ptr(), latitude_deg,
                   out.data_ptr(), out_stride)
        return out
