"""Ensemble MCMC over the fused log-likelihood, on the device.

The reference calibrates SimplyP with emcee's ``EnsembleSampler`` over an IPython.parallel pool
(``Development/2016/MCMC.ipynb:29-31,380``): every half-step of the ensemble copies the walkers to the engines, runs
the model once per walker and copies the log-probabilities back.  :func:`sample` runs the same algorithm — the
affine-invariant stretch move (Goodman & Weare 2010, emcee's default ``StretchMove``) with a uniform prior box — with
the walkers, the random numbers, the proposals and the Metropolis-Hastings test on the GPU
(``simplyp_mcmc_*_device``, ``csrc/simplyp_mcmc.cuh``).  One iteration (per half: propose, integrate the half's
members with the fused statistics, accept) is captured once into a CUDA graph and replayed; the host takes part only
at the start and at the end.

The log-probability of a parameter set is the sum of the Gaussian log-likelihoods of the observed series
(``SIMPLYP_ST_LOGLIK``, ``MCMC.ipynb:213-242``; the error scales ``err_m:<var>`` may be sampled) plus the log of the
unnormalised box prior (0 inside, -inf outside).  A parameter set whose integration raised a status bit gets -inf.
Sampling ``err_phi:<var>`` gives the series of that variable the AR(1) error model of ``simplyp_calibrate_ar1_device``
(autocorrelated residuals, Schoups & Vrugt 2010) with phi sampled alongside the model parameters.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import _cabi
from . import packing as pk

DEFAULT_SEED = 20260101

# p_SC rows the reference checks for an exact sum (f_A + f_S != 1, model.py:318-335): a sampled value would fail it.
_LAND_USE_ROWS = ("f_Ar", "f_IG", "f_S", "f_NC_Ar", "f_NC_IG", "f_NC_S")
# The reference switches the erosion window off for a non-integer day number (``dayNo in np.arange``).
_INTEGER_ONLY = ("d_maxE_spr", "d_maxE_aut")
_SNOW = ("D_snow_0", "f_DDSM")


def _target(name, n_sc, snow_on_device):
    """(kind, index, pos) of the C-ABI for a parameter name of ``ensemble.pack_members``; ValueError if it cannot be
    sampled."""
    if name.startswith(pk.ERR_PHI):
        kind = name[len(pk.ERR_PHI):]
        if kind not in pk.VAR_INDEX:
            raise ValueError("unknown series kind in %r: one of %s" % (name, pk.VAR_KINDS))
        return (_cabi.MCMC_ERROR_MODEL, pk.VAR_INDEX[kind], 0)
    if name.startswith("sc:"):
        row, at = name[3:], None
        if "@" in row:
            row, at = row.split("@", 1)
        if row not in pk.SC_INDEX:
            raise ValueError("unknown sub-catchment parameter %r" % name)
        if row in _LAND_USE_ROWS:
            raise ValueError("%r cannot be sampled: the land-use fractions of a sub-catchment must add to exactly 1" % name)
        if at is None:
            return (_cabi.MCMC_SC_ALL, pk.SC_INDEX[row], 0)
        try:
            pos = int(at)
        except ValueError:
            raise ValueError("bad run-order position in %r" % name) from None
        if not 0 <= pos < n_sc:
            raise ValueError("run-order position of %r outside 0..%d" % (name, n_sc - 1))
        return (_cabi.MCMC_SC_AT, pk.SC_INDEX[row], pos)
    if name not in pk.MEMBER_INDEX:
        raise ValueError("unknown parameter %r" % name)
    if name in _INTEGER_ONLY:
        raise ValueError("%r cannot be sampled: the reference only opens the erosion window on integer days" % name)
    if name in _SNOW and not snow_on_device:
        raise ValueError("%r is only read with snow_on_device=True" % name)
    return (_cabi.MCMC_MEMBER, pk.MEMBER_INDEX[name], 0)


def _check_priors(priors, n_sc, snow_on_device):
    names = list(priors)
    if not names:
        raise ValueError("no free parameters")
    if len(names) > _cabi.MCMC_MAX_FREE:
        raise ValueError("at most %d free parameters" % _cabi.MCMC_MAX_FREE)
    targets = [_target(n, n_sc, snow_on_device) for n in names]
    bounds = np.array([[float(priors[n][0]), float(priors[n][1])] for n in names], dtype=np.float64).reshape(-1, 2)
    for n, (lo, hi) in zip(names, bounds):
        if not (np.isfinite(lo) and np.isfinite(hi)) or not lo < hi:
            raise ValueError("prior of %r needs finite bounds lo < hi, got (%r, %r)" % (n, lo, hi))
    return names, targets, bounds


@dataclass
class McmcResult:
    """What :func:`sample` returns.  ``chain`` [n_saved][W][K] and ``log_prob`` [n_saved][W] hold every ``thin``-th
    iteration (emcee's ``get_chain()`` / ``get_log_prob()`` layout); ``last`` [W][K] / ``last_log_prob`` [W] are the
    walkers after the last iteration; ``iterations`` is the iteration counter after the run (``start_iteration`` +
    ``n_steps``), to be passed as ``start_iteration`` together with ``initial=result`` to continue the run."""
    chain: np.ndarray
    log_prob: np.ndarray
    accepted: np.ndarray
    names: list
    bounds: np.ndarray
    iterations: int
    n_steps: int
    last: np.ndarray
    last_log_prob: np.ndarray

    @property
    def acceptance_fraction(self):
        """Accepted proposals per walker over the iterations of this run."""
        return self.accepted / max(self.n_steps, 1)

    def flat_samples(self, burn=0, thin=1):
        """Stored states after dropping the first ``burn`` stored slots and keeping every ``thin``-th, flattened over
        the walkers: dict name -> array, as ``ensemble.pack_members`` / ``calibrate_ensemble`` /
        ``run_ensemble_to_dir`` take it (posterior predictive runs)."""
        c = self.chain[int(burn)::int(thin)].reshape(-1, len(self.names))
        return {n: np.ascontiguousarray(c[:, k]) for k, n in enumerate(self.names)}


class _Sampler:
    """Device state of one run and the enqueue-only steps of an iteration (used by :func:`sample`)."""

    def __init__(self, met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, priors, n_walkers, n_steps, *,
                 variables=("Q", "TDP"), seed=DEFAULT_SEED, initial=None, start_iteration=0, thin=1, stretch=2.0,
                 step_len=1.0, rtol=None, atol=None, snow_on_device=False, engine=None):
        from .ensemble import latin_hypercube, pack_members
        from .model import make_options

        # ---- host-side validation, before any device work
        n_sc = len(p["SC_list"])
        self.names, targets, self.bounds = _check_priors(priors, n_sc, snow_on_device)
        K, W = len(self.names), int(n_walkers)
        if W % 2 != 0 or W < 2 * K:
            raise ValueError("n_walkers must be even and at least twice the number of free parameters (%d)" % K)
        if int(n_steps) < 1 or int(thin) < 1 or int(start_iteration) < 0:
            raise ValueError("need n_steps >= 1, thin >= 1 and start_iteration >= 0")
        if not float(stretch) > 1.0:
            raise ValueError("the stretch scale must be > 1")
        if initial is None:
            lhs = latin_hypercube(W, {n: tuple(b) for n, b in zip(self.names, self.bounds)}, seed)
            x0 = np.stack([lhs[n] for n in self.names], axis=1)
        elif isinstance(initial, McmcResult):
            if list(initial.names) != self.names:
                raise ValueError("initial result samples %s, not %s" % (initial.names, self.names))
            x0 = initial.last
        elif isinstance(initial, dict):
            x0 = np.stack([np.asarray(initial[n], dtype=np.float64) for n in self.names], axis=1)
        else:
            x0 = np.asarray(initial, dtype=np.float64)
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        if x0.shape != (W, K):
            raise ValueError("initial walkers must have shape (%d, %d), got %s" % (W, K, x0.shape))
        if not np.all((x0 >= self.bounds[:, 0]) & (x0 <= self.bounds[:, 1])):
            raise ValueError("initial walkers must lie inside the prior box")
        p_LU, p_SC = p_LU.copy(deep=True), p_SC.copy(deep=True)
        pk.validate_land_use(p_SC, p["SC_list"])
        pk.check_erosion_windows(p)
        self.topo = pk.build_topology(p_struc, p["SC_list"])
        self.opt = make_options(p_SU, p, dynamic_options, self.topo, step_len, rtol, atol)
        self.opt.snow_on_device = 1 if snow_on_device else 0
        member, sc = pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, self.topo.sc_ids),
                                  {n: x0[:, k] for k, n in enumerate(self.names)})
        obs, desc, self.labels = pk.obs_arrays(obs_dict, self.topo, met_df.index, variables)
        # the AR(1) phi of series v is column phi_col[v] of the walkers (initial evaluation) and of the proposals
        col = pk.ar1_columns(self.names, self.labels, variables)
        self.phi_col = col if any(c >= 0 for c in col) else None
        self.W, self.H, self.K, self.V, self.S = W, W // 2, K, obs.shape[0], n_sc
        self.n_steps, self.thin, self.start = int(n_steps), int(thin), int(start_iteration)
        self.n_saved = (self.start + self.n_steps) // self.thin - self.start // self.thin

        # ---- device state
        import torch
        from .engine import Engine

        self.eng = eng = engine or Engine()
        chain_bytes = 8 * self.n_saved * W * (K + 1)
        if chain_bytes > eng.free_bytes() // 2:
            raise ValueError("the chain needs %.1f GB, more than half of the free device memory: store every n-th "
                             "iteration with thin=n" % (chain_bytes / 1e9))
        dev, f64, i64 = eng.device, torch.float64, torch.int64
        self.d_forc = eng.to_device(pk.forcing_matrix(met_df, raw_snow=bool(snow_on_device)))
        self.d_mem, self.d_sc = eng.to_device(member), eng.to_device(sc)
        self.d_obs, self.d_desc = eng.to_device(obs), eng.to_device(desc)
        self.stats = torch.zeros((W, self.V, pk.NSTAT), dtype=f64, device=dev)
        self.diag = torch.zeros((W, n_sc, pk.NDIAG), dtype=i64, device=dev)
        self.walkers = eng.to_device(x0)
        self.lp = torch.zeros(W, dtype=f64, device=dev)
        self.proposals = torch.zeros((self.H, K), dtype=f64, device=dev)
        self.log_z = torch.zeros(self.H, dtype=f64, device=dev)
        self.out_of_box = torch.zeros(self.H, dtype=torch.int32, device=dev)
        self.iteration = torch.full((1,), self.start, dtype=i64, device=dev)
        self.accepted = torch.zeros(W, dtype=i64, device=dev)
        self.chain = torch.zeros((self.n_saved, W, K), dtype=f64, device=dev)
        self.chain_lp = torch.zeros((self.n_saved, W), dtype=f64, device=dev)
        self.ws_budget = eng.free_bytes() // 2 if self.phi_col is not None else None
        self.mc = _cabi.make_mcmc(W, targets, self.bounds[:, 0], self.bounds[:, 1], n_sc, self.V,
                                  sc_per_member=sc.shape[0] > 1, thin=self.thin, seed=seed, stretch=stretch)
        self.state = _cabi.make_mcmc_state(
            self.walkers.data_ptr(), self.lp.data_ptr(), self.proposals.data_ptr(), self.log_z.data_ptr(),
            self.out_of_box.data_ptr(), self.iteration.data_ptr(), self.accepted.data_ptr(), self.chain.data_ptr(),
            self.chain_lp.data_ptr(), self.n_saved, self.start // self.thin)

    def _stream(self):
        import torch
        return torch.cuda.current_stream(self.eng.device).cuda_stream

    def _rows(self, lo, hi):
        return self.d_mem[lo:hi], (self.d_sc if self.d_sc.shape[0] == 1 else self.d_sc[lo:hi])

    def evaluate_all(self):
        """lp of the current walkers (all W rows in one calibration launch); raises if one is not finite."""
        mem, sc = self._rows(0, self.W)
        with self._device():
            self.diag.zero_()
            self.eng.calibrate(self.d_forc, mem, sc, self.topo.parent_offsets, self.topo.parent_ids, self.d_obs,
                               self.d_desc, self.opt, stats=self.stats, diag=self.diag, **self._phi(self.walkers))
            _cabi.mcmc_init_device(self.mc, self.state, self.stats.data_ptr(), self.diag.data_ptr(), self._stream())
        lp = self.lp.cpu().numpy()
        bad = np.flatnonzero(~np.isfinite(lp))
        if bad.size:
            raise ValueError("the log-probability of initial walker %d is not finite" % bad[0])

    def propose(self, half):
        with self._device():
            _cabi.mcmc_propose_device(self.mc, self.state, half, self.d_mem.data_ptr(), self.d_sc.data_ptr(),
                                      self._stream())

    def evaluate(self, half):
        lo, hi = half * self.H, (half + 1) * self.H
        mem, sc = self._rows(lo, hi)
        with self._device():
            self.diag[lo:hi].zero_()
            self.eng.calibrate(self.d_forc, mem, sc, self.topo.parent_offsets, self.topo.parent_ids, self.d_obs,
                               self.d_desc, self.opt, stats=self.stats[lo:hi], diag=self.diag[lo:hi],
                               **self._phi(self.proposals))

    def _phi(self, rows):
        # the workspace budget is fixed up front: no memory query while an iteration is being captured
        return {} if self.phi_col is None else {"phi": rows, "phi_col": self.phi_col,
                                                "max_workspace_bytes": self.ws_budget}

    def accept(self, half):
        lo = half * self.H
        with self._device():
            _cabi.mcmc_accept_device(self.mc, self.state, half, self.stats[lo].data_ptr(), self.diag[lo].data_ptr(),
                                     self._stream())

    def iteration_step(self):
        """Enqueue one iteration: propose, evaluate, accept for half 0, then for half 1."""
        for half in (0, 1):
            self.propose(half)
            self.evaluate(half)
            self.accept(half)

    def _device(self):
        import torch
        return torch.cuda.device(self.eng.device)

    def capture(self):
        """One iteration captured into a CUDA graph (the iteration counter lives on the device)."""
        import torch
        g = torch.cuda.CUDAGraph()
        with self._device():
            with torch.cuda.graph(g):
                self.iteration_step()
        return g

    def run(self):
        """The first iteration directly (it also loads every kernel), the others as replays of a captured one."""
        self.evaluate_all()
        self.iteration_step()
        if self.n_steps > 1:
            g = self.capture()
            with self._device():
                for _ in range(self.n_steps - 1):
                    g.replay()

    def result(self):
        import torch
        torch.cuda.synchronize(self.eng.device)
        return McmcResult(chain=self.chain.cpu().numpy(), log_prob=self.chain_lp.cpu().numpy(),
                          accepted=self.accepted.cpu().numpy(), names=list(self.names), bounds=self.bounds.copy(),
                          iterations=int(self.iteration.item()), n_steps=self.n_steps,
                          last=self.walkers.cpu().numpy(), last_log_prob=self.lp.cpu().numpy())


def sample(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, priors, n_walkers, n_steps, *,
           variables=("Q", "TDP"), seed=DEFAULT_SEED, initial=None, start_iteration=0, thin=1, stretch=2.0,
           step_len=1.0, rtol=None, atol=None, snow_on_device=False, engine=None):
    """Draw from the posterior of the parameters in ``priors`` with ``n_walkers`` walkers over ``n_steps`` iterations.

    Inputs are those of ``ensemble.calibrate_ensemble``; ``priors`` maps parameter names of
    ``ensemble.pack_members`` (member fields, ``sc:<row>``, ``sc:<row>@<run-order position>``) to the bounds
    ``(lo, hi)`` of a uniform prior (``ensemble.TARLAND_RANGES`` works as it is), and ``err_phi:<var>`` to the box of
    the AR(1) autocorrelation of the residuals of ``var`` (e.g. (0, 0.99)).  The other parameters keep the
    values of ``p`` / ``p_LU`` / ``p_SC``.  ``initial``: walkers [W][K] (or a dict name -> [W], or an
    :class:`McmcResult` to continue, with ``start_iteration=result.iterations``); default: a Latin hypercube over the
    prior box drawn with ``seed``, which also keys the sampler's random numbers.  ``thin``: every ``thin``-th
    iteration is stored.  ``stretch``: the scale a of the stretch move.

    Raises ``ValueError`` before any device work for a name that cannot be sampled — unknown, the integer-valued
    ``d_maxE_*``, the land-use fractions ``sc:f_*``, ``D_snow_0`` / ``f_DDSM`` without ``snow_on_device``, ``err_phi``
    of an unknown variable or of one not among ``variables`` — for bounds
    that are not finite with lo < hi, and for an odd ``n_walkers`` or fewer than twice the free parameters; after the
    initial evaluation, if an initial walker's log-probability is not finite.
    """
    s = _Sampler(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, priors, n_walkers, n_steps,
                 variables=variables, seed=seed, initial=initial, start_iteration=start_iteration, thin=thin,
                 stretch=stretch, step_len=step_len, rtol=rtol, atol=atol, snow_on_device=snow_on_device,
                 engine=engine)
    s.run()
    return s.result()


def autocorr_time(chain, c=5.0):
    """Integrated autocorrelation time per parameter of ``chain`` [n_steps][W][K] (or [n_steps][W], or [n_steps]):
    emcee's estimator — the normalised autocorrelation function of every walker by FFT, averaged over the walkers,
    summed up to the smallest window M with M >= c * tau (Sokal's automatic window)."""
    x = np.asarray(chain, dtype=np.float64)
    if x.ndim == 1:
        x = x[:, None, None]
    elif x.ndim == 2:
        x = x[:, :, None]
    n_t, n_w, n_d = x.shape
    n = 1
    while n < n_t:
        n <<= 1
    tau = np.empty(n_d)
    for d in range(n_d):
        y = x[:, :, d] - x[:, :, d].mean(axis=0)
        f = np.fft.fft(y, n=2 * n, axis=0)
        acf = np.fft.ifft(f * np.conjugate(f), axis=0)[:n_t].real
        acf = (acf / acf[0]).mean(axis=1)
        taus = 2.0 * np.cumsum(acf) - 1.0
        m = np.arange(n_t) < c * taus
        window = int(np.argmin(m)) if np.any(m) else n_t - 1
        tau[d] = taus[window]
    return tau
