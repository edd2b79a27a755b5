"""Timing of the period aggregates (ensemble.period_statistics) on one GPU: one JSON line per case.

Per case the members are integrated in full-output chunks (the chunking of ``period_statistics``), every chunk is
reduced into its columns of the values matrix of each period set, and one selection launch per period set follows;
after one warm-up pass, CUDA events time the phases of a second pass: the chunked integration (``Engine.run``), the
aggregation kernel per period set (with the output columns it reads over its time) and the selection.  The Tarland
2004 case times the route the aggregates replace, ``run_ensemble_to_dir`` (into a temporary directory) and NumPy sums
over the memory-mapped files, with a host clock.  The card's name and power limit are read in the same run.

    python scripts/bench_loads.py [--out lines.jsonl] [--no-old-route]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

Q = (0.025, 0.5, 0.975)
# columns of the raw output a (series, member, day, reach) reads: Qr, Msus, TDP, PP fluxes
_FLUX = {0: set(), 1: {7}, 2: {9}, 3: {11}, 4: {9, 11}, 5: {9}}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def columns_read(desc, n_wb):
    """8-byte output columns read per (member, day), summed over the series."""
    n = 0
    for target, kind, stat in desc:
        cols = _FLUX[kind] | ({5} if (stat != 1 or kind == 0) else set())
        n += len(cols) * (n_wb if target < 0 else 1)
    return n


def tarland_case(st, en, M):
    from simplyp_b200 import ensemble as ens, model as spm, packing as pk, tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(st, en, dynamic="y")
    topo = pk.build_topology(p_struc, p["SC_list"])
    samples = ens.latin_hypercube(M, seed=7)
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), samples)
    series = [(1, v, s) for v in ("Q", "TDP", "TP") for s in ("load", "fwmc", "mean") if not (v, s) == ("Q", "fwmc")]
    desc, _, wb = ens._period_series(series, topo, p_struc)
    return dict(inputs=(met, p_struc, p_SU, p_LU, p_SC, p, dyn), samples=samples, topo=topo, member=member, sc=sc,
                opt=spm.make_options(p_SU, p, dyn, topo), forcing=pk.forcing_matrix(met), dates=met.index,
                desc=desc, wb=wb, series="load, fwmc, mean of Q, TDP, TP at reach 1")


def network_case(M):
    from simplyp_b200 import synthetic
    w = synthetic.scale_config(3, members=M)
    S = w["topo"].n_sc
    w["wb"] = np.array([S - 1, S // 2, S // 4, S // 8, 0], dtype=np.int32)     # five reaches into the water body
    w["desc"] = np.array([(-1, 4, 1), (-1, 2, 2), (-1, 0, 0), (-1, 1, 1), (S - 1, 4, 1), (S - 1, 2, 2)], dtype=np.int32)
    w["dates"] = w["met"].index
    w["series"] = "water body (run-order reaches %s): TP load, TDP fwmc, Q mean, SS load; outlet TP load, TDP fwmc" \
        % w["wb"].tolist()
    return w


def run_case(name, w, M, periods, card, power, chunk=None):
    import torch
    from simplyp_b200 import ensemble as ens, packing as pk
    from simplyp_b200.engine import Engine

    eng = Engine()
    topo, opt = w["topo"], w["opt"]
    S, D = topo.n_sc, w["forcing"].shape[0]
    if chunk is None:                                     # period_statistics' default: about 1 GiB of output a chunk
        chunk = min(M, max(1, (1 << 30) // (S * D * pk.NOUT * 8)))
    sets = [(p,) + tuple(ens.period_bounds(w["dates"], p)) for p in periods]
    d_forc, d_mem, d_sc = eng.to_device(w["forcing"]), eng.to_device(w["member"]), eng.to_device(w["sc"])
    V = w["desc"].shape[0]
    values = [torch.empty((V * len(b), M), dtype=torch.float64, device=eng.device) for _, b, _ in sets]
    out = torch.empty((chunk, S, D, pk.NOUT), dtype=torch.float64, device=eng.device)
    diag = torch.zeros((M, S, pk.NDIAG), dtype=torch.int64, device=eng.device)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def one_pass():
        marks = []
        for m0 in range(0, M, chunk):
            n = min(chunk, M - m0)
            scp = d_sc if d_sc.shape[0] == 1 else d_sc[m0:m0 + n]
            e = [ev() for _ in range(2 + len(sets))]
            e[0].record()
            eng.run(d_forc, d_mem[m0:m0 + n], scp, topo.parent_offsets, topo.parent_ids, opt, out=out[:n],
                    diag=diag[m0:m0 + n])
            e[1].record()
            for k, (_, b, _) in enumerate(sets):
                eng.period_aggregates(out[:n], d_mem[m0:m0 + n], scp, diag[m0:m0 + n], w["desc"], b, w["wb"],
                                      values[k], m0)
                e[2 + k].record()
            marks.append(e)
        sel = []
        for k in range(len(sets)):
            s0, s1 = ev(), ev()
            s0.record()
            eng.nanquantile(values[k], Q)
            s1.record()
            sel.append((s0, s1))
        sel[-1][1].synchronize()
        t_run = sum(e[0].elapsed_time(e[1]) for e in marks)
        t_agg = [sum(e[1 + k].elapsed_time(e[2 + k]) for e in marks) for k in range(len(sets))]
        return t_run, t_agg, [a.elapsed_time(b) for a, b in sel]

    one_pass()                                            # warm-up: module load, workspace
    t_run, t_agg, t_sel = one_pass()
    cols = columns_read(w["desc"], len(w["wb"]))
    line = {"case": name, "gpu": card, "power_limit": power, "members": M, "reaches": S, "days": D, "series": V,
            "series_desc": w["series"], "members_per_chunk": chunk, "chunks": -(-M // chunk),
            "quantiles": list(Q), "ms_integration": round(t_run, 3)}
    for k, (p, b, _) in enumerate(sets):
        covered = int(np.sum(b[:, 1] - b[:, 0] + 1))
        read = 8 * cols * covered * M + 8 * M * S * 4     # output columns of the covered days, the status words
        line.update({"periods_%s" % p: int(len(b)), "ms_aggregate_%s" % p: round(t_agg[k], 3),
                     "aggregate_%s_GB_per_s" % p: round(read / (t_agg[k] * 1e-3) / 1e9, 1),
                     "ms_selection_%s" % p: round(t_sel[k], 3)})
    line["full_output_GB"] = round(8 * pk.NOUT * S * D * M / 1e9, 2)
    return line


def old_route(name, w, M, card, power):
    """run_ensemble_to_dir into a temporary directory, then TP loads per year summed in NumPy over the memory-mapped
    flux files and their quantiles (the route the aggregates replace)."""
    import torch
    from simplyp_b200 import ensemble as ens
    d = tempfile.mkdtemp(prefix="simplyp_loads_bench_")
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ens.run_ensemble_to_dir(*w["inputs"], w["samples"], d)
        t1 = time.perf_counter()
        tdp = np.load(os.path.join(d, "TDP_kg_per_day.npy"), mmap_mode="r")[:, 0, :]
        pp = np.load(os.path.join(d, "PP_kg_per_day.npy"), mmap_mode="r")[:, 0, :]
        diag = np.load(os.path.join(d, "diag.npy"))
        load = np.sum(tdp + pp, axis=1)
        load[np.any(diag[:, :, 3] != 0, axis=1)] = np.nan
        qs = np.nanquantile(load, Q)
        t2 = time.perf_counter()
        disk = sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))
    finally:
        shutil.rmtree(d, True)
    assert qs.shape == (len(Q),)
    return {"case": name + "_old_route", "gpu": card, "power_limit": power, "members": M,
            "series": "TP load at reach 1, one period", "s_run_ensemble_to_dir": round(t1 - t0, 3),
            "s_numpy_sums_and_quantiles": round(t2 - t1, 3), "bytes_on_disk": disk}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", help="also append the lines to this file")
    ap.add_argument("--no-old-route", action="store_true", help="skip the run_ensemble_to_dir + NumPy route")
    a = ap.parse_args()
    from simplyp_b200 import _cabi
    _cabi.require_device()
    card, power = gpu_info()

    def emit(line):
        s = json.dumps(line)
        print(s, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(s + "\n")
    emit(run_case("tarland_2000_2009", tarland_case("2000-01-01", "2009-12-31", 20000), 20000, ("year", "month"),
                  card, power))
    w = tarland_case("2004-01-01", "2004-12-31", 20000)
    emit(run_case("tarland_2004", w, 20000, ("year", "month"), card, power))
    if not a.no_old_route:
        emit(old_route("tarland_2004", w, 20000, card, power))
    # one chunk: 64 members of the 256-reach network are 36 GB of full output
    emit(run_case("config3_waterbody", network_case(64), 64, ("year", "month"), card, power, chunk=64))


if __name__ == "__main__":
    main()
