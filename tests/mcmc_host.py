"""Test-only host build of the ensemble sampler's per-walker arithmetic (simplyp_mcmc.cuh, see mcmc_host.cpp).

The library is compiled with g++ on first use into a temporary directory, so the tests also run from a read-only
tree."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "mcmc_host.cpp")

_lib = None


def load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="simplyp_mcmc_host_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsimplyp_mcmc_host.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def philox(ctr, key):
    """Philox4x32-10 of simplyp_mcmc.cuh: ctr [n][4], key [n][2] (uint32) -> [n][4] uint32."""
    lib = load()
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32).reshape(-1, 4)
    key = np.ascontiguousarray(np.broadcast_to(np.asarray(key, dtype=np.uint32), (ctr.shape[0], 2)))
    out = np.zeros_like(ctr)
    lib.mcmc_host_philox(ctr.ctypes.data_as(C.c_void_p), key.ctypes.data_as(C.c_void_p),
                         out.ctypes.data_as(C.c_void_p), C.c_int(ctr.shape[0]))
    return out


def propose(mc, walkers, t, half):
    """Proposals of one half: (prop [W/2][K], log_z [W/2], out_of_box [W/2])."""
    lib = load()
    walkers = np.ascontiguousarray(walkers, dtype=np.float64)
    H, K = mc.n_walkers // 2, mc.n_free
    prop, log_z = np.zeros((H, K)), np.zeros(H)
    oob = np.zeros(H, dtype=np.int32)
    vp = C.c_void_p
    lib.mcmc_host_propose(C.byref(mc), walkers.ctypes.data_as(vp), C.c_longlong(int(t)), C.c_int(int(half)),
                          prop.ctypes.data_as(vp), log_z.ctypes.data_as(vp), oob.ctypes.data_as(vp))
    return prop, log_z, oob


def accept(mc, t, half, lp_new, log_z, prop, walkers, lp, accepted):
    """Metropolis-Hastings step of one half; updates walkers / lp / accepted in place and returns the decisions
    [W/2]."""
    lib = load()
    H = mc.n_walkers // 2
    lp_new = np.ascontiguousarray(lp_new, dtype=np.float64)
    log_z = np.ascontiguousarray(log_z, dtype=np.float64)
    prop = np.ascontiguousarray(prop, dtype=np.float64)
    for a, dt in ((walkers, np.float64), (lp, np.float64), (accepted, np.int64)):
        assert a.dtype == dt and a.flags["C_CONTIGUOUS"]
    dec = np.zeros(H, dtype=np.int32)
    vp = C.c_void_p
    lib.mcmc_host_accept(C.byref(mc), C.c_longlong(int(t)), C.c_int(int(half)), lp_new.ctypes.data_as(vp),
                         log_z.ctypes.data_as(vp), prop.ctypes.data_as(vp), walkers.ctypes.data_as(vp),
                         lp.ctypes.data_as(vp), accepted.ctypes.data_as(vp), dec.ctypes.data_as(vp))
    return dec
