"""Vertices of the prior box, the matrix of run options and the bound of their comparison with the oracle.

Differential evolution and the sampler propose members on or next to the faces of ``TARLAND_RANGES`` and Sobol'
designs cover the whole box, so the integrator has to agree with the oracle (``oracle/simplyp_oracle.py``, LSODA at
rtol=1e-10) there as well as at the interior points the other parity tests use.  Used by test_box_vertices_cpu.py
(host build of the quad program) and test_box_vertices_gpu.py (the device).
"""
import itertools
import multiprocessing as mp
import os

import numpy as np

from simplyp_b200 import ensemble as ens
from simplyp_b200 import model as spm
from simplyp_b200 import packing as pk
from tests.parity import ATOL, PARITY, RTOL
from tests.util import FLOW_CONC_COLS, max_rel_floored

ORACLE_TOL = dict(rtol=1e-10, atol=1e-13, mxstep=50000)

#: the 5-reach network's own sub-catchment rows, sampled per member (sc_params [M][S][NP_SC])
NETWORK_SC_RANGES = {"sc:A_catch@2": (5.0, 60.0), "sc:L_reach": (2000.0, 20000.0), "sc:S_reach": (0.001, 0.05)}
#: the snow module's parameters (snow_on_device)
SNOW_RANGES = {"D_snow_0": (0.0, 40.0), "f_DDSM": (1.0, 4.0)}

#: Dynamic_EPC0 x Dynamic_erodibility x step_len x run_mode
OPTIONS = list(itertools.product("yn", "yn", (1.0, 0.5), ("cal", "val")))
OPTION_IDS = ["epc0%s-ero%s-step%g-%s" % o for o in OPTIONS]

TARLAND_WINDOW = ("2004-01-01", "2004-12-31")
SNOW_WINDOW = ("2003-10-01", "2004-09-30")        # a whole winter: the pack builds up and melts


def vertices(n, seed, ranges=None):
    """``n`` vertices of the box ``ranges`` (default TARLAND_RANGES) as samples (dict name -> [n]): all parameters at
    their low ends, all at their high ends, then ``n - 2`` vertices drawn with ``seed`` (each end with probability
    1/2)."""
    ranges = ens.TARLAND_RANGES if ranges is None else ranges
    rng = np.random.default_rng(seed)
    high = rng.random((n, len(ranges))) < 0.5
    high[0], high[1] = False, True
    return {k: np.where(high[:, j], hi, lo) for j, (k, (lo, hi)) in enumerate(ranges.items())}


def vertex_label(samples, i):
    """The vertex as a string of L/H, one letter per parameter in the order of ``samples``."""
    out = ""
    for k, v in samples.items():
        lo, hi = {**ens.TARLAND_RANGES, **NETWORK_SC_RANGES, **SNOW_RANGES}[k]
        out += "L" if v[i] == lo else "H"
    return out


def load_case(option, network=False, snow=False):
    """Inputs of one case: (inputs 8-tuple, step_len) with the dynamic options and the run mode of ``option``."""
    from simplyp_b200 import tarland
    from tests.golden.networks import network5_inputs
    epc0, ero, step_len, mode = option
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(*(SNOW_WINDOW if snow else TARLAND_WINDOW), dynamic="y")
    dyn["Dynamic_EPC0"], dyn["Dynamic_erodibility"] = epc0, ero
    p_SU["run_mode"] = mode
    if network:
        p, p_LU, p_SC, p_struc = network5_inputs(p, p_LU, p_SC, p_struc)
    pk.validate_land_use(p_SC, p["SC_list"])
    return (p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs), step_len


class Case:
    """The packed arguments of one launch over all ``samples`` and what the oracle needs for each member."""

    def __init__(self, option, samples, network=False, snow=False):
        inputs, self.step_len = load_case(option, network, snow)
        self.p_SU, self.dyn, self.p, self.p_LU, self.p_SC, self.p_struc, self.met, _obs = inputs
        self.samples, self.snow = samples, snow
        self.topo = pk.build_topology(self.p_struc, self.p["SC_list"])
        self.member, self.sc = ens.pack_members(pk.member_vector(self.p, self.p_LU),
                                                pk.sc_matrix(self.p_SC, self.topo.sc_ids), samples)
        self.raw = self.met[["T_air", "PET", "Precipitation"]]
        self.forcing = pk.forcing_matrix(self.raw, raw_snow=True) if snow else pk.forcing_matrix(self.met)
        self.M = self.member.shape[0]

    def options(self, tighten=1.0):
        opt = spm.make_options(self.p_SU, self.p, self.dyn, self.topo, self.step_len, RTOL / tighten, ATOL / tighten)
        opt.snow_on_device = 1 if self.snow else 0
        return opt

    def run(self, runner, tighten=1.0, members=None):
        """(out, diag) of ``runner`` (hostemu.run_quad or _cabi.run_host) over ``members`` (default: all) in one call."""
        idx = slice(None) if members is None else members
        sc = self.sc[idx] if self.sc.shape[0] > 1 else self.sc
        return runner(self.forcing, self.member[idx], sc, self.topo.parent_offsets, self.topo.parent_ids,
                      self.options(tighten))

    def oracle_args(self, i):
        """Picklable arguments of :func:`oracle_member` for member ``i``: the reference's frames with its values."""
        from simplyp_b200 import inputs as spi
        p, p_LU, p_SC = ens.apply_member_to_pandas(self.samples, i, self.p, self.p_LU, self.p_SC)
        met = self.met
        if self.snow:
            met = spi.snow_hydrol_inputs(float(self.member[i, pk.MEMBER_INDEX["D_snow_0"]]),
                                         float(self.member[i, pk.MEMBER_INDEX["f_DDSM"]]), self.raw)
        return met, self.p_struc, self.p_SU, p_LU, p_SC, p, self.dyn, self.step_len

    def frames(self, out_i, i):
        """{SC: df_R} of member ``i``'s raw block [S][D][25]."""
        R = {}
        for k, SC in enumerate(self.topo.sc_ids):
            A = float(self.sc[i if self.sc.shape[0] > 1 else 0, k, pk.SC_INDEX["A_catch"]])
            _tc, R[SC] = spm.raw_to_frames(out_i[k], self.met.index, A, self.p["Msoil_m2"],
                                           float(self.member[i, pk.MEMBER_INDEX["f_TDP"]]), "None", None)
        return R

    def area(self, i, k):
        return float(self.sc[i if self.sc.shape[0] > 1 else 0, k, pk.SC_INDEX["A_catch"]])


def oracle_member(args):
    """{SC: [D][len(FLOW_CONC_COLS)]} of the oracle for one member (a task of :func:`oracle_runs`)."""
    from oracle import simplyp_oracle as orc
    met, p_struc, p_SU, p_LU, p_SC, p, dyn, step_len = args
    _TC, R, _Kf, _ = orc.run_simply_p(met, p_struc, p_SU, p_LU, p_SC, p, dyn, step_len=step_len, **ORACLE_TOL)
    return {SC: r[FLOW_CONC_COLS].to_numpy(float) for SC, r in R.items()}


def oracle_pool():
    """Worker processes for the oracle (spawned: the parent may hold a CUDA context); close it when done."""
    cores = os.cpu_count() or 1
    return mp.get_context("spawn").Pool(min(cores, 32))


def oracle_runs(pool, case):
    """The oracle on every member of ``case``, one member per task."""
    return pool.map(oracle_member, [case.oracle_args(i) for i in range(case.M)], chunksize=1)


def floors(want, A, f_TDP, rtol=RTOL, atol=ATOL):
    """Per day, the floor of each column of FLOW_CONC_COLS ([D][len(FLOW_CONC_COLS)] ``want``, the reference): the
    value atol/rtol of the daily sum it comes from, carried into the column's units.

    The bound of the comparison is |got - want| <= PARITY (|want| + floor) (util.max_rel_floored).  The integrator
    weighs the error of a state or daily sum y with atol + rtol |y| (simplyp_quad.cuh, as LSODA does); the bound is
    that weight times PARITY/rtol = 100, the margin the 1e-5 relative bound keeps over rtol = 1e-7.  So it is 1e-5
    relative where |y| >> atol/rtol (within 10 % of it above ten floors), and below the floor, where the integrator
    controls absolute error, at most 2 PARITY atol/rtol = 200 atol in the column's units; nothing smaller is asked of
    an integrator run at atol.  The flow and flux columns are daily sums (Qr in mm, Msus / TDP / PP in kg), TP the sum
    of two, SRP f_TDP x TDP, Q_cumecs Qr A 1000/86400 and a concentration flux / (Qr A), with the day's Qr (itself
    relative-controlled: Qr >= Qg_min >> atol/rtol)."""
    c = {k: j for j, k in enumerate(FLOW_CONC_COLS)}
    y0 = atol / rtol
    qa = np.abs(want[:, c["Qr"]]) * A
    per_unit = {"Qr": 1.0, "Q_cumecs": A * 1000.0 / 86400.0, "Msus_kg/day": 1.0, "TDP_kg/day": 1.0, "PP_kg/day": 1.0,
                "TP_kg/day": 2.0, "SRP_kg/day": f_TDP, "SS_mgl": 1.0 / qa, "TDP_mgl": 1.0 / qa, "PP_mgl": 1.0 / qa,
                "TP_mgl": 2.0 / qa, "SRP_mgl": f_TDP / qa}
    out = np.empty_like(want)
    for k, j in c.items():
        out[:, j] = y0 * per_unit[k]
    return out


class Comparison:
    """Worst error of many (member, reach) series against their references under the bound of :func:`check`."""

    def __init__(self, label):
        self.label = label
        self.worst = (0.0, None)               # (max_rel_floored, where): the bound is PARITY
        self.worst_above = (0.0, None)         # (relative error on the days above the floor, where)
        self.needed_convergence = []           # (where, plain relative error under the floor)
        self.failures = []

    def add(self, got, want, fl, where, got_tight=None):
        """``got`` / ``want`` / ``fl``: [D][len(FLOW_CONC_COLS)] series, reference and floors of one (member, reach).
        ``got_tight``: the same member integrated at rtol/100, atol/100 (the convergence leg), or None to skip it."""
        for j, col in enumerate(FLOW_CONC_COLS):
            e = max_rel_floored(got[:, j], want[:, j], fl[:, j])
            above = np.abs(want[:, j]) >= fl[:, j]
            e_above = float(np.max(np.abs(got[above, j] - want[above, j]) / np.abs(want[above, j]), initial=0.0))
            if e > self.worst[0]:
                self.worst = (e, (where, col))
            if e_above > self.worst_above[0]:
                self.worst_above = (e_above, (where, col))
            if not e <= PARITY:                # (NaN included)
                self.failures.append((where, col, e))
            below = ~above
            if not below.any():
                continue
            with np.errstate(divide="ignore", invalid="ignore"):
                plain = float(np.max(np.abs(got[below, j] - want[below, j]) / np.abs(want[below, j])))
            if plain > PARITY:
                self.needed_convergence.append((where, col, plain))
            if got_tight is not None:
                d0 = np.max(np.abs(got[below, j] - want[below, j]) / fl[below, j])
                d1 = np.max(np.abs(got_tight[below, j] - want[below, j]) / fl[below, j])
                if not (d1 < d0 or d0 == 0.0):
                    self.failures.append((where, col, "not closer at rtol/100: %.3e -> %.3e" % (d0, d1)))

    def report(self):
        e, w = self.worst
        ea, wa = self.worst_above
        return ("%s: worst %.2e of the bound's measure (margin %.1fx) at %s; worst relative error above the floor %.2e "
                "(margin %.1fx) at %s; %d series beyond %g relative under the floor" % (self.label, e, PARITY / max(e, 1e-300), w, ea, PARITY / max(ea, 1e-300),
                                               wa, len(self.needed_convergence), PARITY))

    def check(self):
        print(self.report())
        for where, col, plain in self.needed_convergence:
            print("  convergence leg: %s %s (relative %.2e under the floor)" % (where, col, plain))
        assert not self.failures, (self.label, self.failures[:10])


def compare_with_oracle(case, out, want, label, out_tight=None):
    """Every member and reach of ``out`` (a run of ``case``) against the oracle runs ``want``."""
    cmp = Comparison(label)
    for i in range(case.M):
        R = case.frames(out[i], i)
        Rt = case.frames(out_tight[i], i) if out_tight is not None else None
        f_TDP = float(case.member[i, pk.MEMBER_INDEX["f_TDP"]])
        for k, SC in enumerate(case.topo.sc_ids):
            w = want[i][SC]
            fl = floors(w, case.area(i, k), f_TDP)
            cmp.add(R[SC][FLOW_CONC_COLS].to_numpy(float), w, fl, (i, SC, vertex_label(case.samples, i)),
                    Rt[SC][FLOW_CONC_COLS].to_numpy(float) if Rt is not None else None)
    return cmp
