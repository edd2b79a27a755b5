"""Test-only host build of the differential evolution arithmetic (simplyp_de.cuh, see de_host.cpp).

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
SRC = os.path.join(HERE, "de_host.cpp")

_lib = None


def load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="simplyp_de_host_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsimplyp_de_host.so")
        # -ffp-contract=off: the host build must not fuse what the device forms with explicit roundings
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, SRC])
        _lib = C.CDLL(so)
        _lib.de_host_dither.restype = C.c_double
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def dither(de, g):
    return float(load().de_host_dither(C.byref(de), C.c_longlong(g)))


def picks(de, g):
    """[N][4] int32: r0, r1, r2 (-1 for best1bin), fill point of every member at generation g."""
    out = np.zeros((de.n_population, 4), dtype=np.int32)
    load().de_host_picks(C.byref(de), C.c_longlong(g), _ptr(out))
    return out


def trials(de, pop, best, g):
    pop = np.ascontiguousarray(pop, dtype=np.float64)
    out = np.zeros_like(pop)
    load().de_host_trials(C.byref(de), _ptr(pop), C.c_longlong(best), C.c_longlong(g), _ptr(out))
    return out


def scale(de, u):
    u = np.ascontiguousarray(u, dtype=np.float64)
    out = np.zeros_like(u)
    load().de_host_scale(C.byref(de), C.c_longlong(u.shape[0]), _ptr(u), _ptr(out))
    return out


def energy(y, w, diag):
    """y [R][N], w [R], diag [N][S][4] int64 -> [N]."""
    y = np.ascontiguousarray(y, dtype=np.float64)
    w = np.ascontiguousarray(w, dtype=np.float64)
    diag = np.ascontiguousarray(diag, dtype=np.int64)
    out = np.zeros(y.shape[1])
    load().de_host_energy(_ptr(y), C.c_longlong(y.shape[1]), C.c_int(y.shape[0]), _ptr(w), _ptr(diag),
                          C.c_int(diag.shape[1]), _ptr(out))
    return out


def select(e_trial, trial, pop, energy):
    """In place on pop [N][K] and energy [N]; returns the replaced flags [N] bool."""
    N, K = pop.shape
    e_trial = np.ascontiguousarray(e_trial, dtype=np.float64)
    trial = np.ascontiguousarray(trial, dtype=np.float64)
    out = np.zeros(N, dtype=np.int32)
    load().de_host_select(C.c_int(K), C.c_int(N), _ptr(e_trial), _ptr(trial), _ptr(pop), _ptr(energy), _ptr(out))
    return out.astype(bool)
