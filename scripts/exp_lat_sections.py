"""Experiment: where one warp's cycles go, by section of the day loop (-DSP_LAT_PROBE build, simplyp_quad.cuh).

Builds the library with the section probe into a temporary directory (or takes one: --lib), finds the member of the
bench ensemble (config 2, Tarland 2004) with the most step attempts, and integrates it
  (a) alone: 8 copies of it, one warp, so that the warp's lock-step attempts are exactly its own, and
  (b) in the 10^4-member launch, as the bench runs it (cost pilot and planned placement on).
Prints SM cycles per attempt (RHS evaluations, error norm, controller) and per day boundary (end of day, start of the
next), and appends the lines to --out.
usage: python scripts/exp_lat_sections.py [--lib probe.so] [--label text] [--out profiles/r03_lat_sections.txt]"""
import argparse, os, subprocess, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ap = argparse.ArgumentParser()
ap.add_argument("--lib", default=None, help="a library built with -DSP_LAT_PROBE (default: build one from the tree)")
ap.add_argument("--label", default="tree")
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lat_sections.txt"))
ap.add_argument("--members", type=int, default=10000)
args = ap.parse_args()
if args.lib is None:
    import __graft_entry__ as ge
    args.lib = os.path.join(tempfile.mkdtemp(prefix="sp_lat_"), "libsimplyp_b200_probe.so")
    subprocess.check_call([ge._nvcc()] + ge.NVCC_FLAGS + ["-DSP_LAT_PROBE", "-o", args.lib,
                                                          os.path.join(ge.CSRC, "simplyp_kernels.cu")])
os.environ["SIMPLYP_B200_LIB"] = args.lib          # read when _cabi is imported

import numpy as np
import torch
import bench
from simplyp_b200 import model as spm, packing as pk
from simplyp_b200.engine import Engine

eng = Engine(0)
w = bench.build_workload("2004", args.members)
po, pid = w["topo"].parent_offsets, w["topo"].parent_ids
d_forc, d_obs, d_desc = eng.to_device(w["forcing"]), eng.to_device(w["obs_m"]), eng.to_device(w["desc"])
V = w["obs_m"].shape[0]
assert V * pk.NSTAT >= 7, "the probe's seven counters replace the statistics of a member"


def probe(member, sc, pilot):
    opt = spm.make_options(w["p_SU"], w["p"], w["dyn"], w["topo"], 1.0, None, None)
    if not pilot:
        opt.pilot_days = -1
    M = member.shape[0]
    stats = torch.empty((M, V, pk.NSTAT), dtype=torch.float64, device=eng.device)
    diag = torch.zeros((M, 1, pk.NDIAG), dtype=torch.int64, device=eng.device)
    dm, ds = eng.to_device(member), eng.to_device(sc)
    for _ in range(2):                              # the second run is the one read (module loaded, caches warm)
        eng.calibrate(d_forc, dm, ds, po, pid, d_obs, d_desc, opt, stats=stats, diag=diag)
    torch.cuda.synchronize()
    return stats.cpu().numpy().reshape(M, -1)[:, :7], diag[:, 0, 0].cpu().numpy()


def line(what, c):
    it, days = c[5], c[6]
    per_att = c[0:3] / it
    per_day = c[3:5] / days
    return ("%-8s %-34s attempts %5d days %4d | per attempt: rhs %6.0f err %5.0f ctrl %5.0f = %6.0f | "
            "per day boundary: end %6.0f start %6.0f = %6.0f | boundary share %4.1f %%"
            % (args.label, what, it, days, *per_att, per_att.sum(), *per_day, per_day.sum(),
               100.0 * c[3:5].sum() / c[0:5].sum()))


lat_all, steps = probe(w["member"], w["sc"], pilot=True)
h = int(np.argmax(steps))
lines = [line("heaviest member in %d" % args.members, lat_all[h])]
lat_one, _ = probe(np.repeat(w["member"][h:h + 1], 8, axis=0), np.repeat(w["sc"][h:h + 1], 8, axis=0), pilot=False)
lines.insert(0, line("heaviest member alone (8 copies)", lat_one[0]))
dev = torch.cuda.get_device_name(0)
try:
    pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                        capture_output=True, text=True).stdout.strip().splitlines()[0]
except Exception:
    pl = "n/a"
head = "# %s, power limit / max SM clock %s; member %d (%d attempts of its own); SM cycles (clock64)" % (dev, pl, h, steps[h])
print(head)
print("\n".join(lines), flush=True)
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
with open(args.out, "a") as f:
    f.write(head + "\n" + "\n".join(lines) + "\n")
