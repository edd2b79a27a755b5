"""Host packing layer: the reference's pandas parameter objects -> flat fp64 arrays of the C-ABI.

Layouts are the ones declared in ``include/simplyp_b200.h``.  Everything that depends on the
parameters *and* the day (crop cover, EPC0, source coefficients) is derived on the device; this
module only extracts, validates (same exceptions as reference ``model.py:321-335,357``) and lays out.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

# --- member parameter vector (must match the SIMPLYP_P_* enum) -----------------------------------
MEMBER_FIELDS = [
    "f_quick", "alpha", "fc", "beta", "T_g", "Qg_min", "a_Q", "b_Q", "Qr0_init", "Msoil_m2", "Kf", "TDPg",
    "f_TDP", "E_PP", "E_M", "k_M", "d_maxE_spr", "d_maxE_aut",
    "T_s:A", "T_s:S", "SoilPconc:A", "SoilPconc:S", "P_netInput:A", "P_netInput:NC",
    "EPC0_init_mgl:A", "EPC0_init_mgl:S", "C_cover:A", "C_cover:S", "C_cover:IG",
    "C_measures:A", "C_measures:S", "C_measures:IG",
    "err_m:Q", "err_m:SS", "err_m:TDP", "err_m:PP", "err_m:TP", "err_m:SRP",
    "D_snow_0", "f_DDSM",
]
NP_MEMBER = 40
MEMBER_INDEX = {name: i for i, name in enumerate(MEMBER_FIELDS)}

# --- sub-catchment parameter vector (SIMPLYP_SC_* enum) -------------------------------------------
SC_FIELDS = ["A_catch", "f_Ar", "f_IG", "f_S", "f_NC_Ar", "f_NC_IG", "f_NC_S", "f_spr",
             "S_Ar", "S_IG", "S_SN", "L_reach", "S_reach", "TDPeff"]
NP_SC = 16
SC_INDEX = {name: i for i, name in enumerate(SC_FIELDS)}

NF = 4        # forcing columns
NOUT = 25     # raw output columns
NSTAT = 10
NDIAG = 4

ODE_COLS = ["VsA", "VsS", "Vg", "Vr", "Qr_EndOfDay", "Qr", "Msus_EndOfDay", "Msus_kg/day",
            "TDPr_EndOfDay", "TDP_kg/day", "PPr_EndOfDay", "PP_kg/day"]                    # model.py:737-739
NONODE_COLS = ["Qq", "QsA", "QsS", "Qg", "C_cover_A", "EPC0_A_kgmm", "EPC0_NC_kgmm",
               "TDPs_A_kg", "P_labile_A_kg", "conc_TDPs_A_kgmm",
               "TDPs_NC_kgmm", "P_labile_NC_kg", "conc_TDPs_NC_kgmm"]                      # model.py:743-745
RAW_COLS = ODE_COLS + NONODE_COLS

VAR_KINDS = ["Q", "SS", "TDP", "PP", "TP", "SRP"]      # visualise_results.py:401
VAR_INDEX = {v: i for i, v in enumerate(VAR_KINDS)}
STAT_NAMES = ["n", "NSE", "log_NSE", "loglik", "r2", "pbias", "nRMSD", "SSE", "spearman", "reserved"]

DEFAULT_ERR_M = 0.5   # likelihood error scale when the ensemble does not sample it

# ``err_phi:<kind>``: the lag-one autocorrelation phi of the AR(1) error model of the series of that kind
# (simplyp_calibrate_ar1_device).  Not a column of the member vector: it is passed to the likelihood on its own.
ERR_PHI = "err_phi:"


def _f(x):
    try:
        return float(x)
    except (TypeError, ValueError):
        return float("nan")


def parse_upstream(cell):
    """A ``Reach_structure`` cell -> list of upstream SC ids (reference ``model.py:480-487``)."""
    if isinstance(cell, str):
        return [int(x.strip()) for x in cell.split(",")]
    if isinstance(cell, (int, np.integer)):
        return [int(cell)]
    try:
        if not np.isnan(cell):
            return [int(cell)]
    except TypeError:
        pass
    return []


@dataclass
class Topology:
    sc_ids: list                      # run order (p['SC_list'])
    parent_offsets: np.ndarray        # int32 [S+1]
    parent_ids: np.ndarray            # int32 [E], indices into the run order
    upstream: dict = field(default_factory=dict)

    @property
    def n_sc(self):
        return len(self.sc_ids)

    @property
    def n_edges(self):
        return int(self.parent_offsets[-1])


def build_topology(p_struc, sc_list):
    """CSR list of directly-upstream sub-catchments in run order.

    Raises ``KeyError`` when an upstream SC would not have been run yet — the condition under which
    the reference fails at ``model.py:524`` (``df_R_dict[upstream_SC]``).
    """
    sc_ids = [int(s) for s in sc_list]
    pos = {s: i for i, s in enumerate(sc_ids)}
    offsets = [0]
    ids = []
    ups = {}
    for i, s in enumerate(sc_ids):
        u = parse_upstream(p_struc.loc[s, "Upstream_SCs"])
        ups[s] = u
        for up in u:
            if up not in pos or pos[up] >= i:
                raise KeyError(up)
            ids.append(pos[up])
        offsets.append(len(ids))
    return Topology(sc_ids, np.asarray(offsets, dtype=np.int32),
                    np.asarray(ids if ids else [], dtype=np.int32), ups)


def validate_land_use(p_SC, sc_list):
    """Checks and derived rows of reference ``model.py:318-335``; returns {sc: NC_type}."""
    out = {}
    for SC in sc_list:
        f_A = p_SC.loc["f_IG", SC] + p_SC.loc["f_Ar", SC]
        f_NC_A = (p_SC.loc["f_Ar", SC] * p_SC.loc["f_NC_Ar", SC]) + (p_SC.loc["f_NC_IG", SC] * p_SC.loc["f_IG", SC])
        if (f_A + p_SC.loc["f_S", SC]) != 1:
            raise ValueError("Land use proportions do not add to 1 in SC %s" % SC)
        if f_NC_A > 0:
            if p_SC.loc["f_NC_S", SC] > 0:
                raise ValueError("Sub-catchment %s has 2 kinds of newly-converted land;\n"
                                 "                only one permitted (Semi-natural or agricultural, agricultural "
                                 "can be both arable & IG)" % SC)
            nc = "A"
        elif p_SC.loc["f_NC_S", SC] > 0:
            nc = "S"
        else:
            nc = "None"
        out[SC] = nc
    return out


def member_vector(p, p_LU):
    """One member's parameter vector [NP_MEMBER] from the reference's ``p`` Series and ``p_LU`` frame."""
    v = np.zeros(NP_MEMBER)
    for name, i in MEMBER_INDEX.items():
        if name.startswith("err_m:"):
            v[i] = DEFAULT_ERR_M
        elif ":" in name:
            row, col = name.split(":")
            v[i] = _f(p_LU.loc[row, col]) if (row in p_LU.index and col in p_LU.columns) else float("nan")
        else:
            v[i] = _f(p[name]) if name in p.index else float("nan")
    return v


def sc_matrix(p_SC, sc_ids):
    """[S][NP_SC] array from the reference's ``p_SC`` frame (columns = SC ids)."""
    a = np.zeros((len(sc_ids), NP_SC))
    for j, s in enumerate(sc_ids):
        for name, i in SC_INDEX.items():
            a[j, i] = _f(p_SC.loc[name, s])
    return a


def forcing_matrix(met_df, raw_snow=False):
    """[D][4] array: P, PET, day-of-year, T_air (reference ``model.py:497-498,550``).

    ``raw_snow=True`` (for ``SimplypOptions.snow_on_device``): column 0 is the raw ``Precipitation`` and the
    degree-day snow recursion (``inputs.py:159-210``) runs per member on the device."""
    D = len(met_df)
    f = np.zeros((D, NF))
    f[:, 0] = met_df["Precipitation" if raw_snow else "P"].to_numpy(dtype="float64")
    f[:, 1] = met_df["PET"].to_numpy(dtype="float64")
    f[:, 2] = met_df.index.dayofyear.to_numpy(dtype="float64")
    if "T_air" in met_df.columns:
        f[:, 3] = met_df["T_air"].to_numpy(dtype="float64")
    return f


def check_erosion_windows(p):
    """``assert 30 < d_maxE_* < 335`` of reference ``model.py:355-357``."""
    for season in ("spr", "aut"):
        assert (30 < p["d_maxE_%s" % season] < 335), "'d_maxE_%s' must be between 30 and 335" % season


def obs_arrays(obs_dict, topology, date_index, variables=None, min_obs=10):
    """Dense observation matrix for the fused statistics.

    Returns ``(obs [V][D] with NaN, desc [V][2] int32 (sc index, kind), labels [(sc_id, var)])`` for
    every (reach, variable) that has more than ``min_obs`` observations in the run period — the
    reference's ``n_obs > 10`` rule (``visualise_results.py:429-431``).
    """
    rows, desc, labels = [], [], []
    pos = {s: i for i, s in enumerate(topology.sc_ids)}
    for sc_id, df in obs_dict.items():
        if sc_id not in pos:
            continue
        for var in VAR_KINDS:
            if variables is not None and var not in variables:
                continue
            if var not in df.columns:
                continue
            ser = df[var]
            if int(ser.notnull().sum()) <= min_obs:
                continue
            aligned = ser[~ser.index.duplicated()].reindex(date_index)
            rows.append(aligned.to_numpy(dtype="float64"))
            desc.append((pos[sc_id], VAR_INDEX[var]))
            labels.append((sc_id, var))
    D = len(date_index)
    obs = np.asarray(rows, dtype=np.float64).reshape(len(rows), D) if rows else np.zeros((0, D))
    return obs, np.asarray(desc, dtype=np.int32).reshape(len(desc), 2), labels


def ar1_columns(names, labels, variables):
    """``SimplypAr1.col`` of the observed series ``labels`` [(sc_id, variable)]: the position in ``names`` of
    ``err_phi:<variable>``, or -1 (iid likelihood).  Raises ``ValueError`` for an ``err_phi`` name of an unknown kind
    or of a kind not among ``variables`` (None: every kind)."""
    pos = {}
    for j, name in enumerate(names):
        if not name.startswith(ERR_PHI):
            continue
        kind = name[len(ERR_PHI):]
        if kind not in VAR_INDEX:
            raise ValueError("unknown series kind in %r: one of %s" % (name, VAR_KINDS))
        if variables is not None and kind not in variables:
            raise ValueError("%r: %s is not among the calibrated variables %s" % (name, kind, list(variables)))
        pos[kind] = j
    return [pos.get(var, -1) for _sc, var in labels]
