"""Variance-based global sensitivity analysis on the device: Sobol' indices over a Saltelli design.

What SALib's ``sobol.sample`` / ``sobol.analyze`` do, for the parameters a SimplyP user considers calibrating: which of
them control the fit statistics, or the simulated series day by day.  :func:`sobol_indices` writes the design on the
device (``simplyp_sobol_design_device``: unscrambled Sobol' points with the Joe-Kuo direction numbers, SALib's row
order), integrates it — one fused-statistics launch per workspace chunk for objectives, full-output chunks for series
— and computes the first-order, total and optionally second-order indices of every output row with bootstrap
confidence intervals (``simplyp_sobol_indices_device``).  Only the indices come back to the host.
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


def _check_request(n_base, skip, objectives, series, obs_dict, n_boot, conf_level):
    n_base, skip = int(n_base), int(skip)
    if n_base < 2 or n_base & (n_base - 1):
        raise ValueError("n_base must be a power of two >= 2, got %d" % n_base)
    if skip < 0 or skip + n_base > 1 << 32:
        raise ValueError("need skip >= 0 and skip + n_base <= 2^32")
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
    return n_base, skip, objectives


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
    from .ensemble import _band_series, pack_members
    from .mcmc import _check_priors
    from .model import make_options

    n_sc = len(p["SC_list"])
    phi = [n for n in ranges if str(n).startswith(pk.ERR_PHI)]
    if phi:
        raise ValueError("%s: the AR(1) error model is not part of the fit statistics a Sobol' design evaluates" % phi)
    names, targets, bounds = _check_priors(ranges, n_sc, snow_on_device)
    n_base, skip, objectives = _check_request(n_base, skip, objectives, series, obs_dict, n_boot, conf_level)
    topo = pk.build_topology(p_struc, p["SC_list"])
    K, S, D = len(names), topo.n_sc, len(met_df)
    P = 2 * K + 2 if second_order else K + 2
    M = n_base * P
    if series is not None:
        desc, series_labels = _band_series(series, topo)
        V = desc.shape[0]
        labels = [(sc, var, day) for sc, var in series_labels for day in met_df.index]
    else:
        obs, obs_desc, obs_labels = pk.obs_arrays(obs_dict, topo, met_df.index, variables)
        V = obs.shape[0]
        rows, labels = objective_rows(obs_labels, objectives)
    R = len(labels)
    p_LU, p_SC = p_LU.copy(deep=True), p_SC.copy(deep=True)
    pk.validate_land_use(p_SC, p["SC_list"])
    pk.check_erosion_windows(p)
    opt = make_options(p_SU, p, dynamic_options, topo, step_len, rtol, atol)
    opt.snow_on_device = 1 if snow_on_device else 0
    z = statistics.NormalDist().inv_cdf(0.5 + float(conf_level) / 2.0)

    import torch

    from .engine import Engine

    eng = engine or Engine()
    sc_per_member = any(t[0] != _cabi.MCMC_MEMBER for t in targets)
    design_bytes = 8 * M * (pk.NP_MEMBER + (S * pk.NP_SC if sc_per_member else 0))
    need = 8 * R * M + design_bytes
    if need > eng.free_bytes() // 2:
        raise ValueError("the outputs and the design need %.1f GB, more than half of the free device memory: use a "
                         "smaller n_base or fewer rows" % (need / 1e9))
    base_m, base_sc = pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), {})
    dev = eng.device
    d_mem = eng.to_device(base_m).expand(M, pk.NP_MEMBER).contiguous()
    d_sc = eng.to_device(base_sc)
    if sc_per_member:
        d_sc = d_sc.expand(M, S, pk.NP_SC).contiguous()
    sb = _cabi.make_sobol(targets, bounds[:, 0], bounds[:, 1], S, n_base, skip, sc_per_member, second_order)
    d_forc = eng.to_device(pk.forcing_matrix(met_df, raw_snow=bool(snow_on_device)))
    y = torch.empty((R, M), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        eng.sobol_design(sb, d_mem, d_sc)
        if series is None:
            d_obs, d_desc, d_rows = eng.to_device(obs), eng.to_device(obs_desc), eng.to_device(rows)
            stats, diag = eng.calibrate(d_forc, d_mem, d_sc, topo.parent_offsets, topo.parent_ids, d_obs, d_desc, opt)
            eng.sobol_outputs(stats, diag, d_rows, y)
            del stats
        else:
            d_desc = eng.to_device(desc)
            row_bytes = S * D * pk.NOUT * 8
            if members_per_chunk is None:
                members_per_chunk = max(1, (1 << 30) // max(row_bytes, 1))
            chunk = int(max(1, min(int(members_per_chunk), M)))
            out = torch.empty((chunk, S, D, pk.NOUT), dtype=torch.float64, device=dev)
            diag = torch.zeros((M, S, pk.NDIAG), dtype=torch.int64, device=dev)
            for m0 in range(0, M, chunk):
                n = min(chunk, M - m0)
                scp = d_sc if d_sc.shape[0] == 1 else d_sc[m0:m0 + n]
                eng.run(d_forc, d_mem[m0:m0 + n], scp, topo.parent_offsets, topo.parent_ids, opt, out=out[:n],
                        diag=diag[m0:m0 + n])
                eng.predictive_draws(out[:n], d_mem[m0:m0 + n], scp, diag[m0:m0 + n], d_desc, y.view(V, D, M), m0)
            del out
        del d_mem, d_sc
        res = eng.sobol_indices(sb, y, int(n_boot), z, seed)
    torch.cuda.synchronize(dev)
    n_failed = int(np.any(diag.cpu().numpy()[:, :, 3] != 0, axis=1).sum())
    host = {k: v.cpu().numpy() for k, v in res.items()}
    return SobolResult(names=list(names), bounds=bounds, labels=labels, S1=host["S1"], ST=host["ST"],
                       S1_conf=host["S1_conf"], ST_conf=host["ST_conf"], S2=host.get("S2"),
                       S2_conf=host.get("S2_conf"), mean=host["mean"], var=host["var"], n_used=host["n_used"],
                       n_failed=n_failed, n_base=n_base, conf_level=float(conf_level))
