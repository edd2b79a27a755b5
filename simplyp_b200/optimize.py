"""Differential evolution over the fit statistics, on the device: the best single parameter set in a prior box.

The reference's calibration notebook runs "MAP + emcee" (``Development/2016/MCMC.ipynb``): an optimiser finds the
maximum of the posterior, then the walkers start around it.  :func:`differential_evolution` is the first half, what
``scipy.optimize.differential_evolution(updating='deferred', polish=False)`` does — strategies ``best1bin`` and
``rand1bin``, binomial crossover, dithered mutation, scipy's convergence test — with the population, the random
numbers, the trials and the selection on the GPU (``simplyp_de_*_device``, ``csrc/simplyp_de.cuh``).  One generation
(trial, one fused-statistics launch over the whole population, objective rows, selection) is captured once into a
CUDA graph and replayed; the host reads a convergence flag every ``check_every`` replays.

The objective is a weighted sum of fit statistics of the observed series (``sensitivity.OBJECTIVES``), maximised; the
default ``"lp"`` gives the maximum likelihood, which is the MAP under the sampler's uniform prior box.  A parameter
set whose integration raised a status bit, or whose objective is not a number, never enters the population.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import _cabi
from . import packing as pk

DEFAULT_DE_SEED = 20260104
#: Statistics :func:`differential_evolution` may maximise (a signed bias cannot be).
DE_OBJECTIVES = ("NSE", "log_NSE", "loglik", "r2", "nRMSD", "SSE", "lp")
_MIN_POPULATION = {"best1bin": 3, "rand1bin": 4}


def scale(unit, bounds):
    """Parameter values of unit-cube coordinates ``unit`` [..][K] in the boxes ``bounds`` [K][2]: scipy's
    ``_scale_parameters``, every operation rounded on its own, clamped to the box (``de_scale`` of
    ``csrc/simplyp_de.cuh``, bit for bit)."""
    lo, hi = bounds[:, 0], bounds[:, 1]
    v = 0.5 * (lo + hi) + (np.asarray(unit, dtype=np.float64) - 0.5) * np.fabs(lo - hi)
    return np.where(v < lo, lo, np.where(v > hi, hi, v))


def unscale(x, bounds):
    """Unit-cube coordinates of parameter values ``x`` [..][K]: scipy's ``_unscale_parameters``, clipped to [0, 1]
    as scipy clips an initial population."""
    lo, hi = bounds[:, 0], bounds[:, 1]
    u = (np.asarray(x, dtype=np.float64) - 0.5 * (lo + hi)) * (1.0 / np.fabs(lo - hi)) + 0.5
    return np.clip(u, 0.0, 1.0)


def latin_hypercube_unit(n, k, seed):
    """scipy's ``init_population_lhs``: one draw in each of n equal strata per dimension, the strata permuted
    independently per dimension; [n][k] in [0, 1)."""
    rng = np.random.default_rng(seed)
    samples = (1.0 / n) * rng.uniform(size=(n, k)) + np.linspace(0.0, 1.0, n, endpoint=False)[:, None]
    pop = np.zeros_like(samples)
    for j in range(k):
        pop[:, j] = samples[rng.permutation(n), j]
    return pop


def _objective_weights(objective, obs_labels):
    """(rows [R][2] int32, labels, weights [R]) of the objective: a statistic name, or a dict {stat: w} (every
    observed series) / {(sc_id, variable, stat): w} (one series)."""
    from .sensitivity import objective_rows
    obj = {objective: 1.0} if isinstance(objective, str) else objective
    if not isinstance(obj, dict) or not obj:
        raise ValueError("objective must be a statistic name or a non-empty dict of weights")
    stats = []
    for key, w in obj.items():
        stat = key[2] if isinstance(key, tuple) and len(key) == 3 else key
        if stat not in DE_OBJECTIVES:
            raise ValueError("unknown statistic %r: one of %s" % (key, DE_OBJECTIVES))
        if isinstance(key, tuple) and stat != "lp" and (key[0], key[1]) not in obs_labels:
            raise ValueError("unknown series %r: the observed series are %s" % (key[:2], obs_labels))
        if isinstance(w, bool) or not np.isfinite(float(w)):
            raise ValueError("the weight of %r is not a finite number" % (key,))
        if stat not in stats:
            stats.append(stat)
    rows, labels = objective_rows(obs_labels, stats)
    weights = np.array([float(obj.get(lab, 0.0)) + float(obj.get(lab[2], 0.0)) for lab in labels])
    keep = weights != 0.0
    if not keep.any():
        raise ValueError("every objective weight is zero")
    return rows[keep], [lab for lab, k in zip(labels, keep) if k], weights[keep]


@dataclass
class DeResult:
    """What :func:`differential_evolution` returns.  ``best`` (name -> value) is the member of the largest
    ``best_objective`` (the weighted objective; larger is better).  ``population`` [N][K] in parameter units and
    ``objectives`` [N] are the last population; ``unit`` [N][K] is the same population in the unit cube (what a
    continuation starts from).  ``history`` [G][4] holds, after 0, 1, .. generations of this run: the best objective,
    the mean and the standard deviation of the finite objectives, and how many trials replaced their target.
    ``generations`` is the generation counter after the run, to be passed as ``start_generation`` together with
    ``initial=result`` to continue it; ``converged`` whether scipy's test ``std(E) <= tol_abs + tol |mean(E)|`` held
    (at generation ``converged_at``).  ``n_evaluations`` counts the parameter sets integrated, ``n_failed`` those whose
    integration raised a status bit or whose objective was not a number."""
    names: list
    bounds: np.ndarray
    labels: list
    weights: np.ndarray
    best: dict
    best_objective: float
    population: np.ndarray
    objectives: np.ndarray
    unit: np.ndarray
    history: np.ndarray
    generations: int
    converged: bool
    converged_at: object
    n_evaluations: int
    n_failed: int

    def top(self, n):
        """The ``n`` members of the largest objectives (ties: lowest index first) as a dict name -> [n], the form
        ``mcmc.sample(initial=...)`` takes.  A converged population can be nearly degenerate — its members may
        differ in the last digits only — so walkers started from it need many iterations to spread out."""
        n = int(n)
        if not 1 <= n <= self.population.shape[0]:
            raise ValueError("n must lie in 1..%d" % self.population.shape[0])
        order = np.argsort(-self.objectives, kind="stable")[:n]
        return {k: np.ascontiguousarray(self.population[order, j]) for j, k in enumerate(self.names)}


class _Optimizer:
    """Device state of one run and the enqueue-only steps of a generation (used by :func:`differential_evolution`)."""

    def __init__(self, met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population,
                 max_generations, *, objective="lp", variables=("Q", "TDP"), strategy="best1bin", mutation=(0.5, 1.0),
                 recombination=0.7, tol=0.01, tol_abs=0.0, seed=DEFAULT_DE_SEED, initial=None, start_generation=0,
                 check_every=10, step_len=1.0, rtol=None, atol=None, snow_on_device=False, engine=None):
        from .ensemble import pack_members
        from .mcmc import _check_priors
        from .model import make_options

        # ---- host-side validation, before any device work
        n_sc = len(p["SC_list"])
        self.names, targets, self.bounds = _check_priors(ranges, n_sc, snow_on_device)
        K, N = len(self.names), int(n_population)
        if strategy not in _MIN_POPULATION:
            raise ValueError("unknown strategy %r: one of %s" % (strategy, tuple(_MIN_POPULATION)))
        if not _MIN_POPULATION[strategy] <= N < 2 ** 31 - 1:
            raise ValueError("%s needs n_population >= %d" % (strategy, _MIN_POPULATION[strategy]))
        if int(max_generations) < 1 or int(start_generation) < 0 or int(check_every) < 1:
            raise ValueError("need max_generations >= 1, start_generation >= 0 and check_every >= 1")
        m = np.atleast_1d(np.asarray(mutation, dtype=np.float64))
        m = np.array([m[0], m[0]]) if m.size == 1 else m
        if m.size != 2 or not (0.0 <= m[0] <= m[1] < 2.0):
            raise ValueError("mutation must be F or (lo, hi) with 0 <= lo <= hi < 2, got %r" % (mutation,))
        if not 0.0 <= float(recombination) <= 1.0:
            raise ValueError("recombination must lie in [0, 1], got %r" % (recombination,))
        for name, v in (("tol", tol), ("tol_abs", tol_abs)):
            if not (np.isfinite(float(v)) and float(v) >= 0.0):
                raise ValueError("%s must be finite and >= 0, got %r" % (name, v))
        topo = pk.build_topology(p_struc, p["SC_list"])
        obs, desc, obs_labels = pk.obs_arrays(obs_dict, topo, met_df.index, variables)
        rows, self.labels, self.weights = _objective_weights(objective, obs_labels)
        col = pk.ar1_columns(self.names, obs_labels, variables)
        self.phi_col = col if any(c >= 0 for c in col) else None
        if initial is None:
            u0 = latin_hypercube_unit(N, K, seed)
        elif isinstance(initial, DeResult):
            if list(initial.names) != self.names:
                raise ValueError("initial result optimises %s, not %s" % (initial.names, self.names))
            u0 = initial.unit
        else:
            x0 = initial
            if isinstance(initial, dict):
                x0 = np.stack([np.asarray(initial[n], dtype=np.float64) for n in self.names], axis=1)
            x0 = np.asarray(x0, dtype=np.float64)
            if x0.shape != (N, K):
                raise ValueError("initial population must have shape (%d, %d), got %s" % (N, K, x0.shape))
            if not np.all((x0 >= self.bounds[:, 0]) & (x0 <= self.bounds[:, 1])):
                raise ValueError("initial population must lie inside the box")
            u0 = unscale(x0, self.bounds)
        u0 = np.ascontiguousarray(u0, dtype=np.float64)
        if u0.shape != (N, K):
            raise ValueError("initial population must have shape (%d, %d), got %s" % (N, K, u0.shape))
        p_LU, p_SC = p_LU.copy(deep=True), p_SC.copy(deep=True)
        pk.validate_land_use(p_SC, p["SC_list"])
        pk.check_erosion_windows(p)
        self.topo = topo
        self.opt = make_options(p_SU, p, dynamic_options, topo, step_len, rtol, atol)
        self.opt.snow_on_device = 1 if snow_on_device else 0
        member, sc = pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids),
                                  {n: scale(u0, self.bounds)[:, k] for k, n in enumerate(self.names)})
        self.N, self.K, self.V, self.S, self.R = N, K, obs.shape[0], n_sc, rows.shape[0]
        self.max_generations, self.start = int(max_generations), int(start_generation)
        self.check_every = int(check_every)

        # ---- device state
        import torch
        from .engine import Engine

        self.eng = eng = engine or Engine()
        need = 8 * N * (self.V * pk.NSTAT + n_sc * pk.NDIAG + pk.NP_MEMBER + (sc.shape[0] > 1) * n_sc * pk.NP_SC
                        + 2 * K + self.R + 2) + 32 * (self.max_generations + 1)
        if need > eng.free_bytes() // 2:
            raise ValueError("the population needs %.1f GB, more than half of the free device memory: use a smaller "
                             "n_population" % (need / 1e9))
        dev, f64, i64 = eng.device, torch.float64, torch.int64
        self.d_forc = eng.to_device(pk.forcing_matrix(met_df, raw_snow=bool(snow_on_device)))
        self.d_mem, self.d_sc = eng.to_device(member), eng.to_device(sc)
        self.d_obs, self.d_desc = eng.to_device(obs), eng.to_device(desc)
        self.d_rows, self.d_weights = eng.to_device(rows), eng.to_device(self.weights)
        self.stats = torch.zeros((N, self.V, pk.NSTAT), dtype=f64, device=dev)
        self.diag = torch.zeros((N, n_sc, pk.NDIAG), dtype=i64, device=dev)
        self.y = torch.zeros((self.R, N), dtype=f64, device=dev)
        # parameter values of the rows being evaluated: where the AR(1) phi, which no member row holds, is read
        self.values = torch.zeros((N, K), dtype=f64, device=dev) if self.phi_col is not None else None
        self.ws_budget = eng.free_bytes() // 2 if self.phi_col is not None else None
        self.population = eng.to_device(u0)
        self.energy = torch.zeros(N, dtype=f64, device=dev)
        self.trial = torch.zeros((N, K), dtype=f64, device=dev)
        self.flags = torch.zeros(N, dtype=torch.int32, device=dev)
        # generation, best, converged, converged_at, n_failed
        self.counters = torch.tensor([self.start, 0, 0, -1, 0], dtype=i64, device=dev)
        self.history = torch.full((self.max_generations + 1, 4), float("nan"), dtype=f64, device=dev)
        self.de = _cabi.make_de(N, targets, self.bounds[:, 0], self.bounds[:, 1], n_sc, self.R,
                                sc_per_member=sc.shape[0] > 1, strategy=strategy, mutation=m,
                                recombination=recombination, tol=tol, tol_abs=tol_abs, seed=seed)
        c = [self.counters[i].data_ptr() for i in range(5)]
        self.state = _cabi.make_de_state(self.population.data_ptr(), self.energy.data_ptr(), self.trial.data_ptr(),
                                         self.flags.data_ptr(), self.d_weights.data_ptr(), *c,
                                         self.history.data_ptr(), self.max_generations + 1, self.start)

    def _device(self):
        import torch
        return torch.cuda.device(self.eng.device)

    def evaluate(self, unit=None):
        """Zero the status words, integrate all N rows with the fused statistics, take the objective rows.  ``unit``:
        the unit-cube rows the member rows hold (default: the trials), where an AR(1) phi is read."""
        unit = self.trial if unit is None else unit
        with self._device():
            self.diag.zero_()
            phi = {}
            if self.phi_col is not None:
                self.eng.de_scale(self.de, unit, self.values)
                # (a fixed workspace budget: no memory query while a generation is being captured)
                phi = {"phi": self.values, "phi_col": self.phi_col, "max_workspace_bytes": self.ws_budget}
            self.eng.calibrate(self.d_forc, self.d_mem, self.d_sc, self.topo.parent_offsets, self.topo.parent_ids,
                               self.d_obs, self.d_desc, self.opt, stats=self.stats, diag=self.diag, **phi)
            self.eng.sobol_outputs(self.stats, self.diag, self.d_rows, self.y)

    def evaluate_initial(self):
        self.evaluate(self.population)
        self.eng.de_init(self.de, self.state, self.y, self.diag)

    def trial_step(self):
        self.eng.de_trial(self.de, self.state, self.d_mem, self.d_sc)

    def select(self):
        self.eng.de_select(self.de, self.state, self.y, self.diag)

    def generation_step(self):
        """Enqueue one generation: trial, evaluate, select."""
        self.trial_step()
        self.evaluate()
        self.select()

    def capture(self):
        """One generation captured into a CUDA graph (the generation counter lives on the device)."""
        import torch
        g = torch.cuda.CUDAGraph()
        with self._device():
            with torch.cuda.graph(g):
                self.generation_step()
        return g

    def converged(self):
        return bool(self.counters[2].item())

    def run(self):
        """The first generation directly (it also loads every kernel), the others as replays of a captured one; the
        converged flag is read every ``check_every`` replays."""
        self.evaluate_initial()
        self.generation_step()
        left = self.max_generations - 1
        if left < 1:
            return
        g = self.capture()
        with self._device():
            while left > 0:
                n = min(self.check_every, left)
                for _ in range(n):
                    g.replay()
                left -= n
                if left > 0 and self.converged():
                    break

    def result(self):
        import torch
        torch.cuda.synchronize(self.eng.device)
        gen, best, conv, conv_at, n_failed = (int(v) for v in self.counters.cpu().numpy())
        unit = self.population.cpu().numpy()
        pop = scale(unit, self.bounds)
        obj = -self.energy.cpu().numpy()
        run = gen - self.start
        return DeResult(names=list(self.names), bounds=self.bounds.copy(), labels=list(self.labels),
                        weights=self.weights.copy(), best={k: float(pop[best, j]) for j, k in enumerate(self.names)},
                        best_objective=float(obj[best]), population=pop, objectives=obj, unit=unit,
                        history=self.history.cpu().numpy()[:run + 1], generations=gen, converged=bool(conv),
                        converged_at=conv_at if conv else None, n_evaluations=self.N * (run + 1), n_failed=n_failed)


def differential_evolution(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population,
                           max_generations, *, objective="lp", variables=("Q", "TDP"), strategy="best1bin",
                           mutation=(0.5, 1.0), recombination=0.7, tol=0.01, tol_abs=0.0, seed=DEFAULT_DE_SEED,
                           initial=None, start_generation=0, check_every=10, step_len=1.0, rtol=None, atol=None,
                           snow_on_device=False, engine=None):
    """The parameter set of the largest ``objective`` in the box ``ranges``, by differential evolution with
    ``n_population`` members over at most ``max_generations`` generations.

    Inputs are those of ``ensemble.calibrate_ensemble``; ``ranges`` maps parameter names of ``ensemble.pack_members``
    to boxes ``(lo, hi)``, as ``mcmc.sample`` takes them (``ensemble.TARLAND_RANGES`` works as it is), including the
    AR(1) autocorrelations ``err_phi:<var>`` of the likelihood's residuals.  The other parameters keep the values of
    ``p`` / ``p_LU`` / ``p_SC``.

    ``objective``: a statistic of ``DE_OBJECTIVES`` (weight 1 on every observed series of ``variables``; ``"lp"`` is the
    sampler's log-probability, so the default finds the maximum likelihood), or a dict of weights ``{stat: w}`` (every
    observed series) or ``{(sc_id, variable, stat): w}`` (one series); the weighted sum is maximised, so give negative
    weights to statistics to minimise, such as ``SSE`` or ``nRMSD``.  ``strategy``: ``"best1bin"`` or ``"rand1bin"``;
    ``mutation``: F, or ``(lo, hi)`` for a factor drawn once per generation; ``recombination``: the crossover
    probability; ``tol`` / ``tol_abs``: scipy's ``tol`` / ``atol`` (the run stops once the standard deviation of the
    population's objectives is at most ``tol_abs + tol |mean|``).  ``initial``: ``None`` (a Latin hypercube drawn with
    ``seed``, which also keys the random numbers of the generations), a population [N][K] or a dict name -> [N] in
    parameter units, or a :class:`DeResult` with ``start_generation=result.generations`` to continue a run.  The
    result does not depend on ``check_every``, how often the host looks at the convergence flag.

    Raises ``ValueError`` before any device work for everything ``mcmc.sample`` refuses in ``ranges``, an unknown
    strategy, ``n_population`` below 3 (best1bin) or 4 (rand1bin), ``max_generations < 1``, a mutation outside
    0 <= lo <= hi < 2, a recombination outside [0, 1], a negative or non-finite ``tol`` / ``tol_abs``, an unknown
    statistic or series, weights that are all zero or not finite, an ``initial`` of the wrong shape or outside the
    box, ``check_every < 1``, and device buffers needing more than half of the free device memory.
    """
    o = _Optimizer(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population,
                   max_generations, objective=objective, variables=variables, strategy=strategy, mutation=mutation,
                   recombination=recombination, tol=tol, tol_abs=tol_abs, seed=seed, initial=initial,
                   start_generation=start_generation, check_every=check_every, step_len=step_len, rtol=rtol,
                   atol=atol, snow_on_device=snow_on_device, engine=engine)
    o.run()
    return o.result()
