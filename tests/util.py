"""Shared helpers of the test-suite."""
import numpy as np

# columns that are daily flows / concentrations (the quantities north_star's 1e-5 bound is about)
FLOW_CONC_COLS = ["Q_cumecs", "SS_mgl", "TDP_mgl", "PP_mgl", "TP_mgl", "SRP_mgl", "Qr", "Msus_kg/day",
                  "TDP_kg/day", "PP_kg/day", "TP_kg/day", "SRP_kg/day"]


def max_rel(a, b):
    """max |a-b| / |b| over elements where b != 0 (absolute difference where b == 0)."""
    a = np.asarray(a, dtype=float)
    b = np.asarray(b, dtype=float)
    d = np.abs(a - b)
    s = np.abs(b)
    out = np.where(s > 0, d / np.where(s > 0, s, 1.0), d)
    return float(np.nanmax(out)) if out.size else 0.0


def max_rel_floored(a, b, floor):
    """max |a-b| / (|b| + floor): the relative error where |b| >> floor, the absolute error in units of the floor
    where |b| << floor (``floor`` broadcasts against ``b``, e.g. one value per day).  With floor = atol/rtol it is the
    error in units of an integrator's error weight atol + rtol |b|, over rtol."""
    a = np.asarray(a, dtype=float)
    b = np.asarray(b, dtype=float)
    if not b.size:
        return 0.0
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor)))     # a NaN in ``a`` is returned, not skipped


def max_mixed(a, b, rtol, atol_frac=1e-6):
    """max |a-b| / (rtol*|b| + rtol*atol_frac*max|b|): <= 1 means within a mixed abs/rel tolerance.

    Used for quantities that pass through ~0 (soil-water flow just above field capacity): SURVEY.md §7
    asks for a mixed metric there."""
    a = np.asarray(a, dtype=float)
    b = np.asarray(b, dtype=float)
    scale = rtol * np.abs(b) + rtol * atol_frac * max(float(np.nanmax(np.abs(b))), 1e-300)
    return float(np.nanmax(np.abs(a - b) / scale))
