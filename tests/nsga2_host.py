"""Test-only host build of the NSGA-II arithmetic (simplyp_nsga2.cuh, see nsga2_host.cpp).

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
SRC = os.path.join(HERE, "nsga2_host.cpp")

_lib = None


def load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="simplyp_nsga2_host_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsimplyp_nsga2_host.so")
        # -ffp-contract=off: the host build must not fuse what the device forms with explicit roundings
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def picks(ns, g):
    out = np.zeros((ns.n_population // 2, 4), dtype=np.int32)
    load().nsga2_host_picks(C.byref(ns), C.c_longlong(g), _ptr(out))
    return out


def offspring(ns, pop, rank, crowd, g):
    """(children [N][K], decisions [N/2][3 + K]) of every pair at generation g."""
    pop = np.ascontiguousarray(pop, dtype=np.float64)
    rank = np.ascontiguousarray(rank, dtype=np.int32)
    crowd = np.ascontiguousarray(crowd, dtype=np.float64)
    out = np.zeros_like(pop)
    dec = np.zeros((pop.shape[0] // 2, 3 + pop.shape[1]), dtype=np.int32)
    load().nsga2_host_offspring(C.byref(ns), _ptr(pop), _ptr(rank), _ptr(crowd), C.c_longlong(g), _ptr(out),
                                _ptr(dec))
    return out, dec


def orient(ns, y, status):
    y = np.ascontiguousarray(y, dtype=np.float64)
    status = np.ascontiguousarray(status, dtype=np.int32)
    f = np.zeros((y.shape[1], y.shape[0]))
    load().nsga2_host_orient(C.byref(ns), _ptr(y), C.c_longlong(y.shape[1]), _ptr(status), _ptr(f))
    return f


def dominance(f):
    f = np.ascontiguousarray(f, dtype=np.float64)
    n, M = f.shape
    out = np.zeros((n, n), dtype=np.int32)
    load().nsga2_host_dominance(_ptr(f), C.c_longlong(n), C.c_int(M), _ptr(out))
    return out.astype(bool)
