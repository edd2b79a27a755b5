"""Timing of the posterior predictive bands (ensemble.predictive_bands) on one GPU: one JSON line per case.

Per case the members are integrated in full-output chunks (the chunking of ``predictive_bands``), each chunk is turned
into its columns of the draws matrix, and one selection launch follows; after one warm-up pass, CUDA events time each
of the three phases of a second pass: the chunked integration (``Engine.run``), the draw kernel (bytes read from the
full output and written to the draws over its time) and the selection kernel.  The Tarland 2004 case also times the
route through ``run_ensemble_to_dir`` (into a temporary directory) and ``np.nanquantile`` on the memory-mapped
files, with a host clock.  The card's name and power limit are read in the same run.

    python scripts/bench_bands.py [--out lines.jsonl] [--no-old-route]
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

Q = (0.025, 0.25, 0.5, 0.75, 0.975)
SEED = 20260102


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def tarland_case(st, en, M):
    from simplyp_b200 import ensemble as ens, model as spm, packing as pk, tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(st, en, dynamic="y")
    topo = pk.build_topology(p_struc, p["SC_list"])
    samples = ens.latin_hypercube(M, seed=7)
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), samples)
    return dict(inputs=(met, p_struc, p_SU, p_LU, p_SC, p, dyn), samples=samples, topo=topo, member=member, sc=sc,
                opt=spm.make_options(p_SU, p, dyn, topo), forcing=pk.forcing_matrix(met),
                desc=np.array([(0, 0), (0, 2)], dtype=np.int32), series="Q, TDP at reach 1")


def config3_case(M):
    from simplyp_b200 import synthetic
    w = synthetic.scale_config(3, members=M)
    S = w["topo"].n_sc
    reaches = [S - 1, S // 2, S // 4, 0]                  # the outlet and three interior reaches (run order)
    w["desc"] = np.array([(s, k) for s in reaches for k in (0, 2)], dtype=np.int32)
    w["series"] = "Q, TDP at run-order reaches %s" % reaches
    return w


def run_case(name, w, M, obs_error, card, power, chunk=None):
    import torch
    from simplyp_b200 import packing as pk
    from simplyp_b200.engine import Engine

    eng = Engine()
    topo, opt = w["topo"], w["opt"]
    S, D, V = topo.n_sc, w["forcing"].shape[0], w["desc"].shape[0]
    if chunk is None:                                     # predictive_bands' default: about 1 GiB of output a chunk
        chunk = min(M, max(1, (1 << 30) // (S * D * pk.NOUT * 8)))
    d_forc, d_mem, d_sc = eng.to_device(w["forcing"]), eng.to_device(w["member"]), eng.to_device(w["sc"])
    d_desc = eng.to_device(w["desc"])
    draws = torch.empty((V, D, M), dtype=torch.float64, device=eng.device)
    out = torch.empty((chunk, S, D, pk.NOUT), dtype=torch.float64, device=eng.device)
    diag = torch.zeros((M, S, pk.NDIAG), dtype=torch.int64, device=eng.device)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def one_pass():
        t_run = t_draw = 0.0
        marks = []
        for m0 in range(0, M, chunk):
            n = min(chunk, M - m0)
            scp = d_sc if d_sc.shape[0] == 1 else d_sc[m0:m0 + n]
            e = [ev() for _ in range(3)]
            e[0].record()
            eng.run(d_forc, d_mem[m0:m0 + n], scp, topo.parent_offsets, topo.parent_ids, opt, out=out[:n],
                    diag=diag[m0:m0 + n])
            e[1].record()
            eng.predictive_draws(out[:n], d_mem[m0:m0 + n], scp, diag[m0:m0 + n], d_desc, draws, m0, obs_error, SEED)
            e[2].record()
            marks.append(e)
        s0, s1 = ev(), ev()
        s0.record()
        eng.nanquantile(draws.view(V * D, M), Q)
        s1.record()
        s1.synchronize()
        for e in marks:
            t_run += e[0].elapsed_time(e[1])
            t_draw += e[1].elapsed_time(e[2])
        return t_run, t_draw, s0.elapsed_time(s1)

    one_pass()                                            # warm-up: module load, workspace
    t_run, t_draw, t_sel = one_pass()
    bytes_read = 8 * 4 * V * D * M + 8 * M * S * 4       # four columns a (series, day, member), the status words
    bytes_written = 8 * V * D * M
    return {"case": name, "gpu": card, "power_limit": power, "members": M, "reaches": S, "days": D, "series": V,
            "series_desc": w["series"], "members_per_chunk": chunk, "chunks": -(-M // chunk),
            "obs_error": bool(obs_error), "quantiles": list(Q),
            "ms_integration": round(t_run, 3), "ms_draws": round(t_draw, 3), "ms_selection": round(t_sel, 3),
            "draws_GB_per_s": round((bytes_read + bytes_written) / (t_draw * 1e-3) / 1e9, 1),
            "draws_bytes": bytes_written, "bands_bytes": 8 * len(Q) * V * D}


def old_route(name, w, M, card, power):
    """run_ensemble_to_dir into a temporary directory, then Q_cumecs / TDP_mgl rebuilt and np.nanquantile over the
    memory-mapped files (the route the bands replace)."""
    import torch
    from simplyp_b200 import ensemble as ens
    from simplyp_b200 import packing as pk
    d = tempfile.mkdtemp(prefix="simplyp_bands_bench_")
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ens.run_ensemble_to_dir(*w["inputs"], w["samples"], d)
        t1 = time.perf_counter()
        qr = np.load(os.path.join(d, "Qr.npy"), mmap_mode="r")[:, 0, :]
        tdp = np.load(os.path.join(d, "TDP_kg_per_day.npy"), mmap_mode="r")[:, 0, :]
        A = w["sc"][:, 0, pk.SC_INDEX["A_catch"]]
        q_cumecs = qr * A[:, None] * 1000 / 86400
        tdp_mgl = (tdp / qr) / A[:, None]
        diag = np.load(os.path.join(d, "diag.npy"))
        bad = np.any(diag[:, :, 3] != 0, axis=1)
        q_cumecs[bad] = np.nan
        tdp_mgl[bad] = np.nan
        bands = [np.nanquantile(x, Q, axis=0) for x in (q_cumecs, tdp_mgl)]
        t2 = time.perf_counter()
        disk = sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))
    finally:
        shutil.rmtree(d, True)
    assert bands[0].shape == (len(Q), qr.shape[1])
    return {"case": name + "_old_route", "gpu": card, "power_limit": power, "members": M, "series": 2,
            "s_run_ensemble_to_dir": round(t1 - t0, 3), "s_numpy_nanquantile": round(t2 - t1, 3),
            "bytes_on_disk": disk}


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
    w = tarland_case("2004-01-01", "2004-12-31", 20000)
    emit(run_case("tarland_2004", w, 20000, True, card, power))
    if not a.no_old_route:
        emit(old_route("tarland_2004", w, 20000, card, power))
    emit(run_case("tarland_1981_2010", tarland_case("1981-01-01", "2010-12-31", 2048), 2048, True, card, power))
    # one chunk: 64 members of the 256-reach network are 36 GB of full output
    emit(run_case("config3", config3_case(64), 64, True, card, power, chunk=64))

if __name__ == "__main__":
    main()
