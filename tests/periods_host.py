"""Test-only host build of the period aggregates' arithmetic (simplyp_periods.cuh, see periods_host.cpp).

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
SRC = os.path.join(HERE, "periods_host.cpp")

_lib = None


def load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="simplyp_periods_host_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsimplyp_periods_host.so")
        # -ffp-contract=off: the host build must not fuse what the device forms with explicit roundings
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _c(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _sc3(sc, M):
    sc = _c(sc, np.float64)
    return sc if sc.ndim == 3 else sc[None]


def waterbody(out, sc, member, reaches):
    """waterbody_kernel's columns [M][D][11] of out [M][S][D][25]."""
    out, member, sc = _c(out, np.float64), _c(member, np.float64), _sc3(sc, out.shape[0])
    r = _c(reaches, np.int32)
    M, S, D = out.shape[:3]
    wb = np.zeros((M, D, 11))
    load().periods_host_waterbody(_ptr(out), _ptr(sc), _ptr(member), _ptr(r), C.c_int(r.size), C.c_int(M), C.c_int(S),
                                  C.c_int(D), C.c_int(sc.shape[0]), _ptr(wb))
    return wb


def aggregate(out, member, sc, diag, desc, bounds, wb):
    """period_aggregate_kernel's values [V P][M] for out [M][S][D][25], desc [V][3], bounds [P][2], wb reaches."""
    out, member, sc = _c(out, np.float64), _c(member, np.float64), _sc3(sc, out.shape[0])
    diag, desc, bounds, wb = _c(diag, np.int64), _c(desc, np.int32), _c(bounds, np.int32), _c(wb, np.int32)
    M, S, D = out.shape[:3]
    V, P = desc.shape[0], bounds.shape[0]
    values = np.zeros((V * P, M))
    load().periods_host_aggregate(_ptr(out), _ptr(member), _ptr(sc), _ptr(diag), _ptr(desc), C.c_int(V), _ptr(bounds),
                                  C.c_int(P), _ptr(wb), C.c_int(wb.size), C.c_int(M), C.c_int(S), C.c_int(D),
                                  C.c_int(sc.shape[0]), _ptr(values))
    return values
