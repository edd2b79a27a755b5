"""Generates tests/golden/ref_config3.npz and ref_config5.npz: BASELINE configs 3 and 5 at their FULL topology on a
time window the CPU oracle can finish (VERDICT r1, item 1a).

    python tests/golden/make_scale_golden.py [3] [5]

config 3: the seed-3 256-sub-catchment network, first 730 days (2 years) of its 30-year forcing;
config 5: the seed-3 4096-sub-catchment network (all reaches drain to the outlet through 487 levels), first 120 days.
Oracle = oracle/simplyp_oracle.py (the restatement pinned bit-identical to the unmodified reference, tests/
test_oracle_pins.py) run through oracle/parallel.py (the same per-reach calls on all host cores) with scipy's LSODA at
rtol=1e-10, atol=1e-13, mxstep=500000 — LSODA integrates the main-stem reaches with BDF there.  Stored: the 25 raw
columns (model.py:737-745 order) of the outlet, the reaches with the largest estimated rate constant, the deepest
levels and a spread of others; the test runs the whole network on the GPU and compares those reaches.
"""
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import parallel as opar, simplyp_oracle as orc      # noqa: E402
from simplyp_b200 import packing as pk, synthetic                # noqa: E402

WINDOW = {3: 730, 5: 120}
# points of the spread per config.  Config 3 (730 days) keeps its fixture under 1 MB with 4: run-order indices 0, 84,
# 169 and 254, of which 254 is already a deepest reach, so 8 reaches in all.  Config 5: 6 points, 12 reaches in all.
SPREAD = {3: 4, 5: 6}


def sampled_reaches(w, n_extra):
    """Run-order indices: outlet, 3 stiffest by the nominal rate estimate, 2 deepest non-outlet, a spread."""
    topo, sc, member = w["topo"], w["sc"][0], w["member"][0]
    S = topo.n_sc
    po, pid = topo.parent_offsets, topo.parent_ids
    area_up = sc[:, pk.SC_INDEX["A_catch"]].copy()
    lvl = np.zeros(S, dtype=int)
    for s in range(S):
        for e in range(po[s], po[s + 1]):
            area_up[s] += area_up[pid[e]]
            lvl[s] = max(lvl[s], lvl[pid[e]] + 1)
    aQ, bQ = member[pk.MEMBER_INDEX["a_Q"]], member[pk.MEMBER_INDEX["b_Q"]]
    rate = aQ * 86400.0 / sc[:, pk.SC_INDEX["L_reach"]] * (3.0 * area_up / sc[:, pk.SC_INDEX["A_catch"]]) ** bQ / (1 - bQ)
    sel = [S - 1] + list(np.argsort(-rate)[:3]) + list(np.argsort(-lvl)[1:3])
    sel += [int(x) for x in np.linspace(0, S - 2, n_extra).astype(int)]
    out = []
    for s in sel:
        if int(s) not in out:
            out.append(int(s))
    return out, lvl, rate


def main():
    cfgs = [int(a) for a in sys.argv[1:] if a in ("3", "5")] or [3, 5]
    for cfg in cfgs:
        w = synthetic.scale_config(cfg, n_days=WINDOW[cfg])
        met = w["met"]
        p, lu, sc, ups = orc.unpack_pandas(w["p_struc"], w["p_LU"], w["p_SC"], w["p"])
        t0 = time.time()
        raw = opar.run_network_parallel(met["P"].to_numpy(), met["PET"].to_numpy(), met.index.dayofyear.to_numpy(), p, lu,
                                        sc, ups, run_mode="cal", dynamic_EPC0=True, dynamic_erodibility=True,
                                        rtol=1e-10, atol=1e-13, mxstep=500000)
        sel, lvl, rate = sampled_reaches(w, SPREAD[cfg])
        full = np.concatenate([raw["ode"], raw["nonode"]], axis=2)          # [S][D][25]
        path = os.path.join(HERE, "ref_config%d.npz" % cfg)
        np.savez_compressed(path, reaches=np.array(sel, dtype=np.int32), raw=full[sel], levels=lvl[sel],
                            rate_estimate=rate[sel], n_sc=len(raw["sc_ids"]), n_days=len(met),
                            nfe_per_sc_day=raw["nfe"] / (len(raw["sc_ids"]) * len(met)),
                            forcing_head=w["forcing"][:5], rtol=1e-10, atol=1e-13,
                            # daily flow of every reach on the last day: a checksum over the whole network
                            qr_last_day=full[:, -1, 5])
        print("config %d: %d reaches x %d days, %.0f s, %.1f RHS/SC-day, sampled %s (levels %s) -> %s (%d kB)"
              % (cfg, len(raw["sc_ids"]), len(met), time.time() - t0, raw["nfe"] / (len(raw["sc_ids"]) * len(met)), sel,
                 list(lvl[sel]), path, os.path.getsize(path) // 1024), flush=True)


if __name__ == "__main__":
    main()
