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

:func:`nsga2` keeps the statistics apart instead: NSGA-II (Deb et al. 2002) returns the Pareto front of M fit
statistics, the parameter sets for which no series can be fitted better without fitting another one worse.  Offspring,
ranking, crowding and survival run on the GPU (``simplyp_nsga2_*_device``, ``csrc/simplyp_nsga2.cuh``); a generation
is captured once into a CUDA graph and replayed like DE's.  Both optimisers share their setup (:class:`_Search`).
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


class _Search:
    """What both optimisers share: the validation of ``ranges`` and ``initial``, the model inputs, the observed
    series and objective rows, the member rows of the population, the memory check, the device buffers of an
    evaluation and :meth:`evaluate`.  A subclass checks its own options (``_check_options``), names its objective rows
    (``_objective_rows``), counts its own device bytes (``_state_bytes``) and builds its state (``_make_state``)."""

    result_type = None

    def __init__(self, met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population,
                 max_generations, *, variables, seed, initial, start_generation, step_len, rtol, atol, snow_on_device,
                 engine, **options):
        from .ensemble import _model_inputs, pack_members
        from .mcmc import _check_priors

        # ---- host-side validation, before any device work
        n_sc = len(p["SC_list"])
        self.names, self.targets, self.bounds = _check_priors(ranges, n_sc, snow_on_device)
        K, N = len(self.names), int(n_population)
        self.K, self.N = K, N
        self._check_options(max_generations=max_generations, start_generation=start_generation, **options)
        inp = _model_inputs(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, step_len, rtol, atol,
                            snow_on_device)
        self.topo, self.opt = inp.topo, inp.opt
        obs, desc, obs_labels = pk.obs_arrays(obs_dict, self.topo, met_df.index, variables)
        rows = self._objective_rows(obs_labels)
        col = pk.ar1_columns(self.names, obs_labels, variables)
        self.phi_col = col if any(c >= 0 for c in col) else None
        self.initial_result = None
        if initial is None:
            u0 = latin_hypercube_unit(N, K, seed)
        elif isinstance(initial, self.result_type):
            if list(initial.names) != self.names:
                raise ValueError("initial result optimises %s, not %s" % (initial.names, self.names))
            self._check_continuation(initial)
            u0 = initial.unit
            self.initial_result = initial
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
        member, sc = pack_members(inp.member, inp.sc,
                                  {n: scale(u0, self.bounds)[:, k] for k, n in enumerate(self.names)})
        self.V, self.S, self.R = obs.shape[0], n_sc, rows.shape[0]
        self.sc_per_member = sc.shape[0] > 1
        self.max_generations, self.start = int(max_generations), int(start_generation)

        # ---- device state
        import torch
        from .engine import Engine, check_device_memory, half_free_bytes

        self.eng = eng = engine or Engine()
        need = 8 * N * (self.V * pk.NSTAT + n_sc * pk.NDIAG + pk.NP_MEMBER + self.sc_per_member * n_sc * pk.NP_SC
                        + self.R) + self._state_bytes()
        check_device_memory(eng, need, "the population needs", "use a smaller n_population")
        dev, f64, i64 = eng.device, torch.float64, torch.int64
        self.d_forc = eng.to_device(inp.forcing)
        self.d_mem, self.d_sc = eng.to_device(member), eng.to_device(sc)
        self.d_obs, self.d_desc = eng.to_device(obs), eng.to_device(desc)
        self.d_rows = eng.to_device(rows)
        self.stats = torch.zeros((N, self.V, pk.NSTAT), dtype=f64, device=dev)
        self.diag = torch.zeros((N, n_sc, pk.NDIAG), dtype=i64, device=dev)
        self.y = torch.zeros((self.R, N), dtype=f64, device=dev)
        # parameter values of the rows being evaluated: where the AR(1) phi, which no member row holds, is read
        self.values = torch.zeros((N, K), dtype=f64, device=dev) if self.phi_col is not None else None
        self.ws_budget = half_free_bytes(eng) if self.phi_col is not None else None
        self.population = eng.to_device(u0)
        self._make_state()

    def _device(self):
        return self.eng.context()

    def evaluate(self, unit=None):
        """Zero the status words, integrate all N rows with the fused statistics, take the objective rows.  ``unit``:
        the unit-cube rows the member rows hold (default: the candidates of the generation), where an AR(1) phi is
        read."""
        unit = self.candidates if unit is None else unit
        with self._device():
            self.diag.zero_()
            phi = {}
            if self.phi_col is not None:
                self.eng.de_scale(self.box, unit, self.values)
                # (a fixed workspace budget: no memory query while a generation is being captured)
                phi = {"phi": self.values, "phi_col": self.phi_col, "max_workspace_bytes": self.ws_budget}
            self.eng.calibrate(self.d_forc, self.d_mem, self.d_sc, self.topo.parent_offsets, self.topo.parent_ids,
                               self.d_obs, self.d_desc, self.opt, stats=self.stats, diag=self.diag, **phi)
            self.eng.sobol_outputs(self.stats, self.diag, self.d_rows, self.y)

    def _check_continuation(self, result):
        """Refuse a previous result this run cannot continue (called with its names already checked)."""

    def capture(self):
        """One generation captured into a CUDA graph (the generation counter lives on the device)."""
        return self.eng.capture(self.generation_step)


class _Optimizer(_Search):
    """Device state of one run and the enqueue-only steps of a generation (used by :func:`differential_evolution`)."""

    result_type = DeResult

    def __init__(self, met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population,
                 max_generations, *, objective="lp", variables=("Q", "TDP"), strategy="best1bin", mutation=(0.5, 1.0),
                 recombination=0.7, tol=0.01, tol_abs=0.0, seed=DEFAULT_DE_SEED, initial=None, start_generation=0,
                 check_every=10, step_len=1.0, rtol=None, atol=None, snow_on_device=False, engine=None):
        self.objective, self.seed = objective, seed
        super().__init__(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population,
                         max_generations, variables=variables, seed=seed, initial=initial,
                         start_generation=start_generation, step_len=step_len, rtol=rtol, atol=atol,
                         snow_on_device=snow_on_device, engine=engine, strategy=strategy, mutation=mutation,
                         recombination=recombination, tol=tol, tol_abs=tol_abs, check_every=check_every)

    def _check_options(self, max_generations, start_generation, strategy, mutation, recombination, tol, tol_abs,
                       check_every):
        N = self.N
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
        self.strategy, self.mutation, self.recombination = strategy, m, recombination
        self.tol, self.tol_abs, self.check_every = tol, tol_abs, int(check_every)

    def _objective_rows(self, obs_labels):
        rows, self.labels, self.weights = _objective_weights(self.objective, obs_labels)
        return rows

    def _state_bytes(self):
        return 8 * self.N * (2 * self.K + 2) + 32 * (int(self.max_generations) + 1)

    def _make_state(self):
        import torch
        eng, N, K = self.eng, self.N, self.K
        dev, f64, i64 = eng.device, torch.float64, torch.int64
        self.d_weights = eng.to_device(self.weights)
        self.energy = torch.zeros(N, dtype=f64, device=dev)
        self.trial = self.candidates = torch.zeros((N, K), dtype=f64, device=dev)
        self.flags = torch.zeros(N, dtype=torch.int32, device=dev)
        # generation, best, converged, converged_at, n_failed
        self.counters = torch.tensor([self.start, 0, 0, -1, 0], dtype=i64, device=dev)
        self.history = torch.full((self.max_generations + 1, 4), float("nan"), dtype=f64, device=dev)
        self.de = self.box = _cabi.make_de(N, self.targets, self.bounds[:, 0], self.bounds[:, 1], self.S, self.R,
                                           sc_per_member=self.sc_per_member, strategy=self.strategy,
                                           mutation=self.mutation, recombination=self.recombination, tol=self.tol,
                                           tol_abs=self.tol_abs, seed=self.seed)
        c = [self.counters[i].data_ptr() for i in range(5)]
        self.state = _cabi.make_de_state(self.population.data_ptr(), self.energy.data_ptr(), self.trial.data_ptr(),
                                         self.flags.data_ptr(), self.d_weights.data_ptr(), *c,
                                         self.history.data_ptr(), self.max_generations + 1, self.start)

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


DEFAULT_NSGA2_SEED = 20260105
DEFAULT_NSGA2_OBJECTIVES = [(1, "Q", "NSE"), (1, "TP", "NSE"), (1, "SS", "log_NSE")]
#: The sense of every statistic :func:`nsga2` may take: +1 maximised, -1 minimised.
NSGA2_SENSE = {"NSE": 1.0, "log_NSE": 1.0, "loglik": 1.0, "r2": 1.0, "lp": 1.0, "SSE": -1.0, "nRMSD": -1.0}
assert set(NSGA2_SENSE) == set(DE_OBJECTIVES)


def _pareto_objectives(objectives, obs_labels):
    """(rows [M][2] int32, labels [(sc_id, variable, stat)], sense [M]) of the objective list of :func:`nsga2`: rows
    ``(sc_id, variable, stat)`` or bare statistic names, which stand for that statistic of every observed series."""
    from .sensitivity import objective_rows
    if isinstance(objectives, (str, tuple)) or not isinstance(objectives, (list, np.ndarray)):
        raise ValueError("objectives must be a list of (sc_id, variable, statistic) rows or statistic names")
    labels = []
    for o in objectives:
        stat = o[2] if isinstance(o, tuple) and len(o) == 3 else o
        if not isinstance(stat, str) or stat not in DE_OBJECTIVES:
            raise ValueError("unknown statistic %r: one of %s" % (o, DE_OBJECTIVES))
        if not isinstance(o, tuple):
            labels += objective_rows(obs_labels, [stat])[1]
        elif stat == "lp":
            labels.append((None, None, "lp"))
        elif (o[0], o[1]) not in obs_labels:
            raise ValueError("unknown series %r: the observed series are %s" % (o[:2], obs_labels))
        else:
            labels.append(tuple(o))
    if len(set(labels)) != len(labels):
        raise ValueError("repeated objective rows in %s" % (labels,))
    if not 2 <= len(labels) <= _cabi.NSGA2_MAX_OBJECTIVES:
        raise ValueError("NSGA-II needs 2..%d objective rows, got %d" % (_cabi.NSGA2_MAX_OBJECTIVES, len(labels)))
    rows = [(0, -1) if st == "lp" else (obs_labels.index((sc, var)), pk.STAT_NAMES.index(st))
            for sc, var, st in labels]
    return (np.asarray(rows, dtype=np.int32).reshape(-1, 2), labels,
            np.array([NSGA2_SENSE[st] for _, _, st in labels]))


def _objective_name(label):
    sc, var, stat = label
    return stat if stat == "lp" else "%s(%s@%s)" % (stat, var, sc)


@dataclass
class ParetoResult:
    """What :func:`nsga2` returns.  ``labels`` [M] are the objective rows (sc_id, variable, statistic).
    ``population`` [N][K] in parameter units and ``unit`` [N][K] in the unit cube are the last population;
    ``objectives`` [N][M] its statistics as they are (not sign-flipped; NaN rows for members whose integration failed
    or whose statistics are not finite); ``rank`` [N] its non-dominated rank (0 = the first front) and ``crowding`` [N]
    its crowding distance, both within the last survival.  ``history`` [G + 1][2 + M] holds, after 0, 1, .. G
    generations of this run: the size of the first front among the survivors, the number of fronts ranked, and the best
    value of each objective over the feasible survivors. ``generations`` is the generation counter after the run, to
    be passed as ``start_generation`` together with ``initial=result`` to continue it; ``n_evaluations`` counts the
    parameter sets integrated in this run, ``n_failed`` those that were infeasible.
    """
    names: list
    bounds: np.ndarray
    labels: list
    population: np.ndarray
    unit: np.ndarray
    objectives: np.ndarray
    rank: np.ndarray
    crowding: np.ndarray
    history: np.ndarray
    generations: int
    n_evaluations: int
    n_failed: int

    def front(self):
        """The members of the first front as a DataFrame: one column per parameter, then one per objective
        (``"NSE(Q@1)"``, ``"lp"``), in population order."""
        import pandas as pd
        f = self.rank == 0
        cols = {k: self.population[f, j] for j, k in enumerate(self.names)}
        cols.update({_objective_name(lab): self.objectives[f, m] for m, lab in enumerate(self.labels)})
        return pd.DataFrame(cols)

    def front_samples(self):
        """The members of the first front as a dict name -> [n], the form ``ensemble.calibrate_ensemble``,
        ``predictive_bands`` and ``period_statistics`` take: what the trade-off means for the simulated series."""
        f = self.rank == 0
        return {k: np.ascontiguousarray(self.population[f, j]) for j, k in enumerate(self.names)}


class _Nsga2(_Search):
    """Device state of one NSGA-II run and the enqueue-only steps of a generation (used by :func:`nsga2`)."""

    result_type = ParetoResult

    def __init__(self, met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population,
                 max_generations, *, objectives=DEFAULT_NSGA2_OBJECTIVES, variables=("Q", "SS", "TP"), crossover=0.9,
                 eta_c=15.0, mutation=None, eta_m=20.0, seed=DEFAULT_NSGA2_SEED, initial=None, start_generation=0,
                 step_len=1.0, rtol=None, atol=None, snow_on_device=False, engine=None):
        self.objective_spec, self.seed = objectives, seed
        super().__init__(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population,
                         max_generations, variables=variables, seed=seed, initial=initial,
                         start_generation=start_generation, step_len=step_len, rtol=rtol, atol=atol,
                         snow_on_device=snow_on_device, engine=engine, crossover=crossover, eta_c=eta_c,
                         mutation=mutation, eta_m=eta_m)

    def _check_options(self, max_generations, start_generation, crossover, eta_c, mutation, eta_m):
        N = self.N
        if N % 2 != 0 or not 4 <= N <= 1 << 29:
            raise ValueError("n_population must be even and >= 4, got %d" % N)
        if int(max_generations) < 1 or int(start_generation) < 0:
            raise ValueError("need max_generations >= 1 and start_generation >= 0")
        for name, v in (("crossover", crossover), ("mutation", 1.0 / self.K if mutation is None else mutation)):
            if isinstance(v, bool) or not 0.0 <= float(v) <= 1.0:
                raise ValueError("%s must lie in [0, 1], got %r" % (name, v))
        for name, v in (("eta_c", eta_c), ("eta_m", eta_m)):
            if not (np.isfinite(float(v)) and float(v) >= 0.0):
                raise ValueError("%s must be finite and >= 0, got %r" % (name, v))
        self.rates = dict(crossover=float(crossover), mutation=mutation, eta_c=float(eta_c), eta_m=float(eta_m))

    def _check_continuation(self, result):
        """A continued run keeps the result's objectives, ranks and crowding without evaluating them again, so the
        objective rows and the boxes must be the result's."""
        if [tuple(lab) for lab in result.labels] != self.labels:
            raise ValueError("initial result has the objectives %s, not %s" % (result.labels, self.labels))
        if not np.array_equal(np.asarray(result.bounds, dtype=np.float64), self.bounds):
            raise ValueError("initial result was run in other boxes: %s, not %s"
                             % (np.asarray(result.bounds).tolist(), self.bounds.tolist()))

    def _objective_rows(self, obs_labels):
        rows, self.labels, self.sense = _pareto_objectives(self.objective_spec, obs_labels)
        self.M = len(self.labels)
        return rows

    def _state_bytes(self):
        """The device bytes of the run's state (and the SimplypNsga2 they follow from)."""
        self.ns = _cabi.make_nsga2(self.N, self.targets, self.bounds[:, 0], self.bounds[:, 1], self.S, self.sense,
                                   sc_per_member=self.sc_per_member, seed=self.seed, **self.rates)
        self.ws_bytes = _cabi.nsga2_workspace_bytes(self.ns)
        return 8 * self.N * (2 * self.K + self.M + 2) + 8 * (int(self.max_generations) + 1) * (2 + self.M) \
            + self.ws_bytes

    def _make_state(self):
        import torch
        eng, N, K, M = self.eng, self.N, self.K, self.M
        dev, f64, i64 = eng.device, torch.float64, torch.int64
        r = self.initial_result
        self.objectives = torch.full((N, M), float("nan"), dtype=f64, device=dev) if r is None \
            else eng.to_device(r.objectives, np.float64)
        self.rank = torch.zeros(N, dtype=torch.int32, device=dev) if r is None else eng.to_device(r.rank, np.int32)
        self.crowding = torch.zeros(N, dtype=f64, device=dev) if r is None else eng.to_device(r.crowding, np.float64)
        self.offspring = self.candidates = torch.zeros((N, K), dtype=f64, device=dev)
        self.counters = torch.tensor([self.start, 0], dtype=i64, device=dev)   # generation, n_failed
        self.history = torch.full((self.max_generations + 1, 2 + M), float("nan"), dtype=f64, device=dev)
        if r is not None:   # a continued run starts where the last one ended, with no evaluation of its own
            self.history[0] = eng.to_device(r.history[-1], np.float64)
        self.workspace = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        # the boxes of the targets, for simplyp_de_scale_device (the AR(1) phi of the rows being evaluated)
        self.box = _cabi.make_de(N, self.targets, self.bounds[:, 0], self.bounds[:, 1], self.S, self.R,
                                 sc_per_member=self.sc_per_member)
        self.state = _cabi.make_nsga2_state(self.population.data_ptr(), self.objectives.data_ptr(),
                                            self.rank.data_ptr(), self.crowding.data_ptr(), self.offspring.data_ptr(),
                                            self.counters[0].data_ptr(), self.counters[1].data_ptr(),
                                            self.history.data_ptr(), self.max_generations + 1,
                                            self.workspace.data_ptr(), self.ws_bytes, self.start)

    def evaluate_initial(self):
        """Evaluate and rank the initial population (nothing for a continued run, whose state is the result's)."""
        if self.initial_result is None:
            self.evaluate(self.population)
            self.eng.nsga2_init(self.ns, self.state, self.y, self.diag)

    def offspring_step(self):
        self.eng.nsga2_offspring(self.ns, self.state, self.d_mem, self.d_sc)

    def survive(self):
        self.eng.nsga2_survive(self.ns, self.state, self.y, self.diag)

    def generation_step(self):
        """Enqueue one generation: offspring, evaluate, survive."""
        self.offspring_step()
        self.evaluate()
        self.survive()

    def run(self):
        """The first generation directly (it also loads every kernel), the others as replays of a captured one."""
        self.evaluate_initial()
        self.generation_step()
        if self.max_generations > 1:
            g = self.capture()
            with self._device():
                for _ in range(self.max_generations - 1):
                    g.replay()

    def result(self):
        import torch
        torch.cuda.synchronize(self.eng.device)
        gen, n_failed = (int(v) for v in self.counters.cpu().numpy())
        unit = self.population.cpu().numpy()
        run = gen - self.start
        return ParetoResult(names=list(self.names), bounds=self.bounds.copy(), labels=list(self.labels),
                            population=scale(unit, self.bounds), unit=unit, objectives=self.objectives.cpu().numpy(),
                            rank=self.rank.cpu().numpy(), crowding=self.crowding.cpu().numpy(),
                            history=self.history.cpu().numpy()[:run + 1], generations=gen,
                            n_evaluations=self.N * (run + (self.initial_result is None)), n_failed=n_failed)


def nsga2(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population, max_generations, *,
          objectives=DEFAULT_NSGA2_OBJECTIVES, variables=("Q", "SS", "TP"), crossover=0.9, eta_c=15.0, mutation=None,
          eta_m=20.0, seed=DEFAULT_NSGA2_SEED, initial=None, start_generation=0, step_len=1.0, rtol=None, atol=None,
          snow_on_device=False, engine=None):
    """The Pareto front of several fit statistics in the box ``ranges``, by NSGA-II (Deb et al. 2002) with
    ``n_population`` members over ``max_generations`` generations: the parameter sets for which no objective can be
    improved without making another one worse.

    Inputs are those of :func:`differential_evolution`; ``ranges`` takes the same boxes, including ``sc:`` rows and the
    AR(1) autocorrelations ``err_phi:<var>``.  ``objectives``: a list of M >= 2 rows ``(sc_id, variable, stat)`` or bare
    statistic names (that statistic of every observed series of ``variables``), statistics of ``DE_OBJECTIVES``; the
    default is ``DEFAULT_NSGA2_OBJECTIVES``.  NSE, log_NSE, loglik, r2 and lp are maximised, SSE and nRMSD minimised
    (``NSGA2_SENSE``).  Variation is in the unit cube: SBX with probability
    ``crossover`` per pair and index ``eta_c``, then polynomial mutation with probability ``mutation`` per variable
    (None: 1/K) and index ``eta_m``.  The run has no convergence test: it takes ``max_generations`` generations.
    ``initial``: ``None`` (a Latin hypercube drawn with ``seed``, which also keys the random numbers of the
    generations), a population [N][K] or a dict name -> [N] in parameter units, or a :class:`ParetoResult` with
    ``start_generation=result.generations`` to continue a run bit for bit.

    Raises ``ValueError`` before any device work for everything :func:`differential_evolution` refuses in ``ranges``,
    an odd ``n_population`` or one below 4, ``max_generations < 1``, ``start_generation < 0``, fewer than 2 or more than
    16 objective rows, an unknown statistic or series, a repeated objective row, ``crossover`` or ``mutation`` outside
    [0, 1], ``eta_c`` or ``eta_m`` negative or not finite, an ``initial`` of the wrong shape or outside the box, an
    initial result with other parameters, objective rows or boxes, and device buffers needing more than half of the
    free device memory.
    """
    o = _Nsga2(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, ranges, n_population, max_generations,
               objectives=objectives, variables=variables, crossover=crossover, eta_c=eta_c, mutation=mutation,
               eta_m=eta_m, seed=seed, initial=initial, start_generation=start_generation, step_len=step_len,
               rtol=rtol, atol=atol, snow_on_device=snow_on_device, engine=engine)
    o.run()
    return o.result()
