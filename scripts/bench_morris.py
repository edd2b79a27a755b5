"""Timing of the Morris screening (sensitivity.elementary_effects) on one GPU: one JSON line per case.

Per case, after one warm-up pass, CUDA events time the phases of a second pass: the selection of optimised
trajectories (cases with a candidate pool), the design kernel, the integration (one fused-statistics
``Engine.calibrate`` for objectives; chunked ``Engine.run`` for series), the outputs kernel or the draw kernel, the
effects entry point with n_boot = 0 (elementary effects and point statistics) and the whole effects entry point with
the bootstrap (its difference to the former is the bootstrap).  Beside them, a host NumPy restatement of the
estimators and the bootstrap runs on the same Y over the first rows, its per-row time scaled to all rows; for the pool
case the NumPy selection runs on the first 512 candidates, its time scaled by the square of the pool ratio (the
all-pairs pass).  The card's name and power limit are read in the same run.

    python scripts/bench_morris.py [--out lines.jsonl] [--host-rows 2]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 20261022
OBJ = ["NSE", "log_NSE", "loglik", "r2", "pbias", "nRMSD", "SSE", "lp"]


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def host_effects(y, lev, p, picks):
    """NumPy restatement of the point statistics and the bootstrap of one row (all trajectories finite)."""
    r, P, K = lev.shape
    Y = y.reshape(r, P)
    d = np.diff(lev, axis=1)
    j = np.argmax(d != 0, axis=2)
    sign = np.sign(np.take_along_axis(d, j[..., None], axis=2)[..., 0])
    ee = np.empty((r, K))
    np.put_along_axis(ee, j, sign * np.diff(Y, axis=1) / (p / (2.0 * (p - 1))), axis=1)
    mu, mu_star, sigma = ee.mean(axis=0), np.abs(ee).mean(axis=0), ee.std(axis=0, ddof=1)
    boot = np.abs(ee)[picks].mean(axis=1)
    return mu, mu_star, sigma, boot.std(axis=0, ddof=1)


def tarland_case(years):
    from simplyp_b200 import ensemble as ens, model as spm, packing as pk, tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(years[0], years[1], dynamic="y")
    topo = pk.build_topology(p_struc, p["SC_list"])
    base_m, base_sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), {})
    return dict(met=met, obs=obs, topo=topo, opt=spm.make_options(p_SU, p, dyn, topo), member=base_m, sc=base_sc,
                forcing=pk.forcing_matrix(met), desc=np.array([(0, 0), (0, 2)], dtype=np.int32))


def network_case():
    from simplyp_b200 import synthetic
    w = synthetic.scale_config(3, members=1)
    w["desc"] = np.array([(w["topo"].n_sc - 1, 0)], dtype=np.int32)     # Q at the outlet
    return w


def run_case(name, w, r, n_candidates, kind, n_boot, card, power, host_rows, chunk_bytes=1 << 30):
    import torch
    from simplyp_b200 import _cabi, ensemble as ens, mcmc, packing as pk
    from simplyp_b200.engine import Engine
    from tests import morris_reference as ref
    eng = Engine()
    topo, opt = w["topo"], w["opt"]
    names, targets, bounds = mcmc._check_priors(ens.TARLAND_RANGES, topo.n_sc, False)
    K, S, D, p = len(names), topo.n_sc, w["forcing"].shape[0], 4
    M = r * (K + 1)
    mo = _cabi.make_morris(targets, bounds[:, 0], bounds[:, 1], S, r, p, n_candidates, True, SEED)
    d_forc = eng.to_device(w["forcing"])
    d_mem = eng.to_device(w["member"][:1]).expand(M, pk.NP_MEMBER).contiguous()
    d_sc = eng.to_device(w["sc"].reshape(1, S, pk.NP_SC)).expand(M, S, pk.NP_SC).contiguous()    # sc:TDPeff
    if kind == "objectives":
        o, odesc, labels = pk.obs_arrays(w["obs"], topo, w["met"].index, ("Q", "TDP"))
        d_obs, d_odesc = eng.to_device(o), eng.to_device(odesc)
        rows = [(v, pk.STAT_NAMES.index(s)) for v in range(len(labels)) for s in OBJ if s != "lp"] + [(0, -1)]
        d_rows = eng.to_device(np.asarray(rows, dtype=np.int32))
        R = len(rows)
    else:
        d_desc = eng.to_device(w["desc"])
        V = w["desc"].shape[0]
        R = V * D
        chunk = int(min(M, max(1, chunk_bytes // (S * D * pk.NOUT * 8))))
        out = torch.empty((chunk, S, D, pk.NOUT), dtype=torch.float64, device=eng.device)
        diag = torch.zeros((M, S, pk.NDIAG), dtype=torch.int64, device=eng.device)
    y = torch.empty((R, M), dtype=torch.float64, device=eng.device)
    z = statistics.NormalDist().inv_cdf(0.975)
    sel = torch.empty(r, dtype=torch.int32, device=eng.device) if n_candidates else None

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def one_pass():
        e = [ev() for _ in range(7)]
        e[0].record()
        if sel is not None:
            eng.morris_select(mo, sel)
        e[1].record()
        eng.morris_design(mo, d_mem, d_sc, sel)
        e[2].record()
        if kind == "objectives":
            stats, dg = eng.calibrate(d_forc, d_mem, d_sc, topo.parent_offsets, topo.parent_ids, d_obs, d_odesc, opt)
            e[3].record()
            eng.sobol_outputs(stats, dg, d_rows, y)
            e[4].record()
            times = None
        else:
            t_run, t_draw = 0.0, 0.0
            diag.zero_()
            for m0 in range(0, M, chunk):
                n = min(chunk, M - m0)
                c = [ev() for _ in range(3)]
                c[0].record()
                eng.run(d_forc, d_mem[m0:m0 + n], d_sc[m0:m0 + n], topo.parent_offsets, topo.parent_ids, opt,
                        out=out[:n], diag=diag[m0:m0 + n])
                c[1].record()
                eng.predictive_draws(out[:n], d_mem[m0:m0 + n], d_sc[m0:m0 + n], diag[m0:m0 + n], d_desc,
                                     y.view(V, D, M), m0)
                c[2].record()
                torch.cuda.synchronize()
                t_run += c[0].elapsed_time(c[1])
                t_draw += c[1].elapsed_time(c[2])
            e[3].record()
            e[4].record()
            times = (t_run, t_draw)
        eng.morris_effects(mo, y, 0, z, sel)
        e[5].record()
        res = eng.morris_effects(mo, y, n_boot, z, sel)
        e[6].record()
        torch.cuda.synchronize()
        if times is None:
            times = (e[2].elapsed_time(e[3]), e[3].elapsed_time(e[4]))
        point, total = e[4].elapsed_time(e[5]), e[5].elapsed_time(e[6])
        return dict(selection_ms=e[0].elapsed_time(e[1]) if sel is not None else None,
                    design_ms=e[1].elapsed_time(e[2]), integration_ms=times[0], outputs_ms=times[1],
                    effects_ms=point, effects_with_bootstrap_ms=total, bootstrap_ms=total - point), res

    one_pass()
    t, res = one_pass()
    selected = sel.cpu().numpy() if sel is not None else np.arange(r)
    lev = ref.levels(SEED, K, p, int(selected.max()) + 1)[selected]
    yh = y[:host_rows].cpu().numpy()
    from tests import morris_host
    picks = morris_host.picks(SEED, n_boot, r)
    h0 = time.perf_counter()
    worst = 0.0
    for i in range(host_rows):
        mu, mu_star, sigma, conf = host_effects(yh[i], lev, p, picks)
        worst = max(worst, float(np.nanmax(np.abs(mu_star - res["mu_star"][i].cpu().numpy()))),
                    float(np.nanmax(np.abs(conf * z - res["mu_star_conf"][i].cpu().numpy()))))
    host_s = (time.perf_counter() - h0) / host_rows * R
    line = dict(case=name, card=card, power_limit=power, K=K, n_trajectories=r, n_candidates=n_candidates,
                members=M, reaches=S, days=D, rows=R, n_boot=n_boot, n_used_min=int(res["n_used"].min().item()),
                **{k: (round(v, 3) if v is not None else None) for k, v in t.items()},
                host_numpy_effects_s_scaled=round(host_s, 3), host_rows_timed=host_rows,
                host_vs_device_max_abs_diff_mu_star_and_conf=worst)
    if n_candidates:
        sub = 512
        h0 = time.perf_counter()
        ref.select(ref.levels(SEED, K, p, sub), r)
        line["host_numpy_selection_s_scaled"] = round((time.perf_counter() - h0) * (n_candidates / sub) ** 2, 1)
        line["host_numpy_selection_candidates_timed"] = sub
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--host-rows", type=int, default=2)
    a = ap.parse_args()
    card, power = gpu_info()
    t04 = tarland_case(("2004-01-01", "2004-12-31"))
    cases = [("tarland2004_objectives_r1000", t04, 1000, 0, "objectives", 1000, {}),
             ("tarland2004_objectives_pool4096_r50", t04, 50, 4096, "objectives", 1000, {}),
             ("tarland1981_2010_series_Q_TDP_r100", tarland_case(("1981-01-01", "2010-12-31")), 100, 0, "series",
              1000, {}),
             ("network256_30y_series_Q_outlet_r20", network_case(), 20, 0, "series", 1000,
              dict(chunk_bytes=40 << 30))]
    lines = []
    for name, w, r, nc, kind, n_boot, kw in cases:
        line = run_case(name, w, r, nc, kind, n_boot, card, power, a.host_rows, **kw)
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
