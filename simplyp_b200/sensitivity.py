"""Global sensitivity analysis on the device: Sobol' indices over a Saltelli design, and Morris screening.

What SALib's ``sobol.sample`` / ``sobol.analyze`` do, for the parameters a SimplyP user considers calibrating: which of
them control the fit statistics, or the simulated series day by day.  :func:`sobol_indices` writes the design on the
device (``simplyp_sobol_design_device``: unscrambled Sobol' points with the Joe-Kuo direction numbers, SALib's row
order), integrates it — one fused-statistics launch per workspace chunk for objectives, full-output chunks for series
— and computes the first-order, total and optionally second-order indices of every output row with bootstrap
confidence intervals (``simplyp_sobol_indices_device``).  Only the indices come back to the host.

:func:`elementary_effects` is the screening step before them, SALib's ``morris.sample`` / ``morris.analyze``: r (K + 1)
members instead of thousands times K, and :meth:`MorrisResult.screen` hands the parameters that matter to the
sampler, the optimisers and :func:`sobol_indices` as a ``ranges`` dict.
"""
from __future__ import annotations

import statistics
from dataclasses import dataclass

import numpy as np

from . import _cabi
from . import packing as pk

DEFAULT_SOBOL_SEED = 20260103
#: Statistics a row may take (``packing.STAT_NAMES``), and ``lp``, the sampler's log-probability of a member.
OBJECTIVES = ("NSE", "log_NSE", "loglik", "r2", "pbias", "nRMSD", "SSE", "lp")


@dataclass
class SobolResult:
    """What :func:`sobol_indices` returns.  Row r of the outputs is ``labels[r]``: (sc_id, variable, statistic) for
    objectives (``(None, None, "lp")`` for the log-probability), (sc_id, variable, date) for series.  ``S1``, ``ST``
    and their ``*_conf`` are [R][K]; ``S2`` and ``S2_conf`` [R][K][K] (NaN outside j < k, None without second order);
    ``mean`` and ``var`` [R] the mean of the used outputs and the variance of the A and B outputs; ``n_used`` [R] the
    samples whose P outputs were all finite; ``n_failed`` the design members whose integration raised a status bit."""
    names: list
    bounds: np.ndarray
    labels: list
    S1: np.ndarray
    ST: np.ndarray
    S1_conf: np.ndarray
    ST_conf: np.ndarray
    S2: object
    S2_conf: object
    mean: np.ndarray
    var: np.ndarray
    n_used: np.ndarray
    n_failed: int
    n_base: int
    conf_level: float

    def table(self, row=0):
        """Per-parameter DataFrame of row ``row`` (an index or a label): S1, S1_conf, ST, ST_conf."""
        import pandas as pd
        r = row if isinstance(row, (int, np.integer)) else self.labels.index(tuple(row))
        return pd.DataFrame({"S1": self.S1[r], "S1_conf": self.S1_conf[r], "ST": self.ST[r],
                             "ST_conf": self.ST_conf[r]}, index=list(self.names))


def objective_rows(obs_labels, objectives):
    """Rows of ``simplyp_sobol_outputs_device`` for the statistics ``objectives`` (names of ``OBJECTIVES``) of the
    observed series ``obs_labels`` [(sc_id, variable)]: (rows [R][2] int32 = (series, ``packing.STAT_NAMES`` slot, or
    -1 for lp), labels [(sc_id, variable, statistic)], ``(None, None, "lp")`` for lp, last)."""
    rows, labels = [], []
    for v, (sc, var) in enumerate(obs_labels):
        for o in objectives:
            if o != "lp":
                rows.append((v, pk.STAT_NAMES.index(o)))
                labels.append((sc, var, o))
    if "lp" in objectives:
        rows.append((0, -1))
        labels.append((None, None, "lp"))
    return np.asarray(rows, dtype=np.int32).reshape(-1, 2), labels


def _check_outputs(objectives, series, obs_dict, n_boot, conf_level):
    """The checks of the outputs and of the bootstrap that sobol_indices and elementary_effects share; returns the
    objectives as a list (or None)."""
    if (objectives is None) == (series is None):
        raise ValueError("give exactly one of objectives and series")
    if objectives is not None:
        if obs_dict is None:
            raise ValueError("objectives need obs_dict")
        objectives = list(objectives)
        if not objectives:
            raise ValueError("no objectives: give statistics among %s" % (OBJECTIVES,))
        for o in objectives:
            if o not in OBJECTIVES:
                raise ValueError("unknown statistic %r: one of %s" % (o, OBJECTIVES))
    if isinstance(n_boot, bool) or int(n_boot) != n_boot or not 0 <= int(n_boot) <= 10000:
        raise ValueError("n_boot must be an integer in 0..10^4, got %r" % (n_boot,))
    if not 0.0 < float(conf_level) < 1.0:
        raise ValueError("conf_level must lie in (0, 1), got %r" % (conf_level,))
    return objectives


def _check_request(n_base, skip, objectives, series, obs_dict, n_boot, conf_level):
    n_base, skip = int(n_base), int(skip)
    if n_base < 2 or n_base & (n_base - 1):
        raise ValueError("n_base must be a power of two >= 2, got %d" % n_base)
    if skip < 0 or skip + n_base > 1 << 32:
        raise ValueError("need skip >= 0 and skip + n_base <= 2^32")
    return n_base, skip, _check_outputs(objectives, series, obs_dict, n_boot, conf_level)


def _check_ranges(ranges, n_sc, snow_on_device, what):
    """``mcmc._check_priors`` of ``ranges`` without the AR(1) error-model parameters, which no design evaluates."""
    from .mcmc import _check_priors
    phi = [n for n in ranges if str(n).startswith(pk.ERR_PHI)]
    if phi:
        raise ValueError("%s: the AR(1) error model is not part of the fit statistics a %s evaluates" % (phi, what))
    return _check_priors(ranges, n_sc, snow_on_device)


def _output_rows(met_df, topo, obs_dict, objectives, series, variables):
    """Labels of the output rows and what :func:`_evaluate` needs to fill them."""
    from .ensemble import _band_series
    if series is not None:
        desc, series_labels = _band_series(series, topo)
        labels = [(sc, var, day) for sc, var in series_labels for day in met_df.index]
        return labels, dict(desc=desc)
    obs, obs_desc, obs_labels = pk.obs_arrays(obs_dict, topo, met_df.index, variables)
    rows, labels = objective_rows(obs_labels, objectives)
    return labels, dict(obs=obs, obs_desc=obs_desc, rows=rows)


def _evaluate(eng, inp, out_rows, d_mem, d_sc, y, members_per_chunk):
    """Integrates the design rows d_mem / d_sc and writes their outputs y [R][M]: one fused-statistics launch per
    workspace chunk and the objective rows, or full-output chunks and their simulated series.  Returns the diag."""
    from .ensemble import _integrate_in_chunks
    topo, opt = inp.topo, inp.opt
    d_forc = eng.to_device(inp.forcing)
    if "desc" not in out_rows:
        d_obs, d_desc, d_rows = (eng.to_device(out_rows[k]) for k in ("obs", "obs_desc", "rows"))
        stats, diag = eng.calibrate(d_forc, d_mem, d_sc, topo.parent_offsets, topo.parent_ids, d_obs, d_desc, opt)
        eng.sobol_outputs(stats, diag, d_rows, y)
        return diag
    d_desc = eng.to_device(out_rows["desc"])
    draws = y.view(d_desc.shape[0], -1, y.shape[1])

    def draw(out, mem, scp, diag, m0):
        eng.predictive_draws(out, mem, scp, diag, d_desc, draws, m0)
    return _integrate_in_chunks(eng, d_forc, d_mem, d_sc, topo, opt, members_per_chunk, draw)


def _design_rows(eng, inp, targets, M, S):
    """Device design rows [M] holding the base parameter vectors; per-member SC rows when a target needs them."""
    from .ensemble import pack_members
    sc_per_member = any(t[0] != _cabi.MCMC_MEMBER for t in targets)
    base_m, base_sc = pack_members(inp.member, inp.sc, {})
    d_mem = eng.to_device(base_m).expand(M, pk.NP_MEMBER).contiguous()
    d_sc = eng.to_device(base_sc)
    if sc_per_member:
        d_sc = d_sc.expand(M, S, pk.NP_SC).contiguous()
    return d_mem, d_sc


def sobol_indices(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, ranges, n_base, *, obs_dict=None,
                  objectives=None, series=None, variables=("Q", "TDP"), second_order=False, n_boot=1000,
                  conf_level=0.95, seed=DEFAULT_SOBOL_SEED, skip=0, members_per_chunk=None, step_len=1.0, rtol=None,
                  atol=None, snow_on_device=False, engine=None):
    """Sobol' first-order (S1), total (ST) and, with ``second_order``, second-order (S2) indices of the parameters in
    ``ranges`` (name -> (lo, hi), the names and boxes ``mcmc.sample`` takes; ``ensemble.TARLAND_RANGES`` works as it
    is), from a Saltelli design of ``n_base`` samples (n_base (K + 2) members, n_base (2K + 2) with second order)
    starting at Sobol' point ``skip``.  The other parameters keep the values of ``p`` / ``p_LU`` / ``p_SC``.

    The outputs are either ``objectives``, fit statistics (``OBJECTIVES``) of every observed series of
    ``variables`` in ``obs_dict``, one row per (series, statistic), plus the row ``lp`` if asked; or ``series``,
    simulated series [(sc_id, variable)] as ``ensemble.predictive_bands`` takes them, one row per (series, day),
    integrated in full-output chunks of ``members_per_chunk`` members.  The estimators are SALib's (Saltelli 2010,
    Jansen 1999, Saltelli 2002); a sample enters a row when all of its P outputs are finite, so a member whose
    integration failed removes its sample.  Confidences are ``z(conf_level)`` times the standard deviation over
    ``n_boot`` bootstrap resamples drawn with ``seed``.

    Raises ``ValueError`` before any device work for everything ``mcmc.sample`` refuses in ``ranges``, the AR(1)
    error-model parameters ``err_phi:*``, an
    ``n_base`` that is not a power of two >= 2, skip + n_base > 2^32, both or neither of ``objectives`` and
    ``series``, objectives without ``obs_dict`` or unknown, a bad series, ``n_boot`` outside 0..10^4, ``conf_level``
    outside (0, 1), and outputs plus design rows needing more than half of the free device memory.
    """
    from .ensemble import _model_inputs, _n_failed

    n_sc = len(p["SC_list"])
    names, targets, bounds = _check_ranges(ranges, n_sc, snow_on_device, "Sobol' design")
    n_base, skip, objectives = _check_request(n_base, skip, objectives, series, obs_dict, n_boot, conf_level)
    inp = _model_inputs(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, step_len, rtol, atol, snow_on_device)
    topo = inp.topo
    K, S = len(names), topo.n_sc
    P = 2 * K + 2 if second_order else K + 2
    M = n_base * P
    labels, out_rows = _output_rows(met_df, topo, obs_dict, objectives, series, variables)
    R = len(labels)
    z = statistics.NormalDist().inv_cdf(0.5 + float(conf_level) / 2.0)

    import torch

    from .engine import Engine, check_device_memory

    eng = engine or Engine()
    sc_per_member = any(t[0] != _cabi.MCMC_MEMBER for t in targets)
    design_bytes = 8 * M * (pk.NP_MEMBER + (S * pk.NP_SC if sc_per_member else 0))
    check_device_memory(eng, 8 * R * M + design_bytes, "the outputs and the design need",
                        "use a smaller n_base or fewer rows")
    dev = eng.device
    d_mem, d_sc = _design_rows(eng, inp, targets, M, S)
    sb = _cabi.make_sobol(targets, bounds[:, 0], bounds[:, 1], S, n_base, skip, sc_per_member, second_order)
    y = torch.empty((R, M), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        eng.sobol_design(sb, d_mem, d_sc)
        diag = _evaluate(eng, inp, out_rows, d_mem, d_sc, y, members_per_chunk)
        del d_mem, d_sc
        res = eng.sobol_indices(sb, y, int(n_boot), z, seed)
    torch.cuda.synchronize(dev)
    n_failed = _n_failed(diag)
    host = {k: v.cpu().numpy() for k, v in res.items()}
    return SobolResult(names=list(names), bounds=bounds, labels=labels, S1=host["S1"], ST=host["ST"],
                       S1_conf=host["S1_conf"], ST_conf=host["ST_conf"], S2=host.get("S2"),
                       S2_conf=host.get("S2_conf"), mean=host["mean"], var=host["var"], n_used=host["n_used"],
                       n_failed=n_failed, n_base=n_base, conf_level=float(conf_level))


# ------------------------------------------------------------------------------------------ Morris screening
DEFAULT_MORRIS_SEED = 20261022
#: Largest candidate pool of the optimised trajectories (``SIMPLYP_MORRIS_MAX_CANDIDATES``).
MAX_CANDIDATES = _cabi.MORRIS_MAX_CANDIDATES


@dataclass
class MorrisResult:
    """What :func:`elementary_effects` returns.  Row r of the outputs is ``labels[r]``, as in :class:`SobolResult`.
    ``mu``, ``mu_star``, ``sigma`` and ``mu_star_conf`` are [R][K]; ``n_used`` [R] the trajectories whose K + 1
    outputs were all finite; ``n_failed`` the design members whose integration raised a status bit; ``selected`` the
    candidate index of every trajectory (0..r-1 without a candidate pool); ``ranges`` the ``ranges`` of the run."""
    names: list
    bounds: np.ndarray
    labels: list
    mu: np.ndarray
    mu_star: np.ndarray
    sigma: np.ndarray
    mu_star_conf: np.ndarray
    n_used: np.ndarray
    n_failed: int
    selected: np.ndarray
    num_levels: int
    conf_level: float
    ranges: dict

    def table(self, row=0):
        """Per-parameter DataFrame of row ``row`` (an index or a label): mu, mu_star, sigma, mu_star_conf."""
        import pandas as pd
        r = row if isinstance(row, (int, np.integer)) else self.labels.index(tuple(row))
        return pd.DataFrame({"mu": self.mu[r], "mu_star": self.mu_star[r], "sigma": self.sigma[r],
                             "mu_star_conf": self.mu_star_conf[r]}, index=list(self.names))

    def screen(self, fraction=0.1, rows=None):
        """The sub-dict of ``ranges``, in its order, of the parameters whose mu_star reaches ``fraction`` times the
        largest mu_star of at least one of ``rows`` (indices or labels; default all rows).  A row whose largest
        mu_star is not a positive number (too few used trajectories, or an output no parameter moves) selects
        nothing.  ``mcmc.sample``, ``optimize.differential_evolution``, ``optimize.nsga2`` and :func:`sobol_indices`
        take the result as it is."""
        if not 0.0 <= float(fraction) <= 1.0:
            raise ValueError("fraction must lie in [0, 1], got %r" % (fraction,))
        idx = range(len(self.labels)) if rows is None else [
            r if isinstance(r, (int, np.integer)) else self.labels.index(tuple(r)) for r in rows]
        keep = np.zeros(len(self.names), dtype=bool)
        for r in idx:
            ms = self.mu_star[r]
            top = np.nanmax(ms) if np.any(np.isfinite(ms)) else np.nan
            if top > 0.0:
                keep |= ms >= float(fraction) * top
        return {n: self.ranges[n] for k, n in enumerate(self.names) if keep[k]}


def _check_morris(n_trajectories, num_levels, n_candidates):
    if isinstance(n_trajectories, bool) or int(n_trajectories) != n_trajectories or int(n_trajectories) < 2:
        raise ValueError("n_trajectories must be an integer >= 2, got %r" % (n_trajectories,))
    r = int(n_trajectories)
    if isinstance(num_levels, bool) or int(num_levels) != num_levels or num_levels % 2 or not 2 <= num_levels <= 16:
        raise ValueError("num_levels must be an even integer in 2..16, got %r" % (num_levels,))
    if n_candidates is not None:
        if (isinstance(n_candidates, bool) or int(n_candidates) != n_candidates
                or not r < int(n_candidates) <= MAX_CANDIDATES):
            raise ValueError("n_candidates must be an integer in n_trajectories + 1 .. %d, got %r"
                             % (MAX_CANDIDATES, n_candidates))
        n_candidates = int(n_candidates)
    return r, int(num_levels), n_candidates or 0


def elementary_effects(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, ranges, n_trajectories, *,
                       obs_dict=None, objectives=None, series=None, variables=("Q", "TDP"), num_levels=4,
                       n_candidates=None, n_boot=1000, conf_level=0.95, seed=DEFAULT_MORRIS_SEED,
                       members_per_chunk=None, step_len=1.0, rtol=None, atol=None, snow_on_device=False,
                       engine=None):
    """Morris elementary effects (mu, mu_star, sigma and a bootstrap confidence of mu_star) of the parameters in
    ``ranges`` (name -> (lo, hi), the names and boxes ``mcmc.sample`` takes) from ``n_trajectories`` one-at-a-time
    trajectories on a grid of ``num_levels`` levels: n_trajectories (K + 1) members.  The other parameters keep the
    values of ``p`` / ``p_LU`` / ``p_SC``.  With ``n_candidates``, the trajectories are the ``n_trajectories`` of
    that many candidates that a greedy search for Campolongo's spread criterion picks (Ruano et al. 2012; not SALib's
    routine); without, trajectory i is candidate i.  DESIGN.md §4h gives the design and the random streams.

    The outputs are those of :func:`sobol_indices`: ``objectives`` (fit statistics of every observed series of
    ``variables`` in ``obs_dict``, and ``lp``) or ``series`` (one row per simulated series and day, integrated in
    full-output chunks of ``members_per_chunk`` members).  A trajectory enters a row when its K + 1 outputs are all
    finite, so a member whose integration failed removes its trajectory.  ``mu_star_conf`` is ``z(conf_level)``
    times the standard deviation of mu_star over ``n_boot`` bootstrap resamples of the used trajectories.
    :meth:`MorrisResult.screen` returns the ``ranges`` worth keeping.

    Raises ``ValueError`` before any device work for everything ``mcmc.sample`` refuses in ``ranges``, the AR(1)
    error-model parameters ``err_phi:*``, ``n_trajectories`` < 2, ``num_levels`` odd or outside 2..16,
    ``n_candidates`` <= ``n_trajectories`` or above ``MAX_CANDIDATES``, what :func:`sobol_indices` refuses in the
    outputs, ``n_boot`` and ``conf_level``, and outputs plus design rows needing more than half of the free device
    memory.
    """
    from .ensemble import _model_inputs, _n_failed

    n_sc = len(p["SC_list"])
    names, targets, bounds = _check_ranges(ranges, n_sc, snow_on_device, "Morris design")
    r, num_levels, n_candidates = _check_morris(n_trajectories, num_levels, n_candidates)
    objectives = _check_outputs(objectives, series, obs_dict, n_boot, conf_level)
    inp = _model_inputs(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, step_len, rtol, atol, snow_on_device)
    topo = inp.topo
    K, S = len(names), topo.n_sc
    M = r * (K + 1)
    labels, out_rows = _output_rows(met_df, topo, obs_dict, objectives, series, variables)
    R = len(labels)
    z = statistics.NormalDist().inv_cdf(0.5 + float(conf_level) / 2.0)

    import torch

    from .engine import Engine, check_device_memory

    eng = engine or Engine()
    sc_per_member = any(t[0] != _cabi.MCMC_MEMBER for t in targets)
    design_bytes = 8 * M * (pk.NP_MEMBER + (S * pk.NP_SC if sc_per_member else 0))
    check_device_memory(eng, 8 * R * M + design_bytes, "the outputs and the design need",
                        "use fewer trajectories or fewer rows")
    dev = eng.device
    mo = _cabi.make_morris(targets, bounds[:, 0], bounds[:, 1], S, r, num_levels, n_candidates, sc_per_member, seed)
    d_mem, d_sc = _design_rows(eng, inp, targets, M, S)
    y = torch.empty((R, M), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        sel = eng.morris_select(mo) if n_candidates else None
        eng.morris_design(mo, d_mem, d_sc, sel)
        diag = _evaluate(eng, inp, out_rows, d_mem, d_sc, y, members_per_chunk)
        del d_mem, d_sc
        res = eng.morris_effects(mo, y, int(n_boot), z, sel)
    torch.cuda.synchronize(dev)
    host = {k: v.cpu().numpy() for k, v in res.items()}
    selected = sel.cpu().numpy().astype(np.int64) if sel is not None else np.arange(r, dtype=np.int64)
    return MorrisResult(names=list(names), bounds=bounds, labels=labels, mu=host["mu"], mu_star=host["mu_star"],
                        sigma=host["sigma"], mu_star_conf=host["mu_star_conf"], n_used=host["n_used"],
                        n_failed=_n_failed(diag), selected=selected, num_levels=num_levels,
                        conf_level=float(conf_level), ranges={n: ranges[n] for n in names})
