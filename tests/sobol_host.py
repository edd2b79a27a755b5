"""Test-only host build of the sensitivity analysis' design and bootstrap arithmetic (simplyp_sobol.cuh, see
sobol_host.cpp).

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
SRC = os.path.join(HERE, "sobol_host.cpp")

_lib = None


def load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="simplyp_sobol_host_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsimplyp_sobol_host.so")
        # -ffp-contract=off: the host build must not fuse what the device forms with explicit roundings
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def table():
    """The embedded direction numbers [128][32] uint32."""
    out = np.zeros((128, 32), dtype=np.uint32)
    load().sobol_host_table(_ptr(out))
    return out


def points(D, n, skip=0):
    """Points skip .. skip + n - 1 [n][D] uint32."""
    out = np.zeros((n, D), dtype=np.uint32)
    load().sobol_host_points(C.c_int(D), C.c_int64(n), C.c_int64(skip), _ptr(out))
    return out


def design(sb, member_offset, n):
    """Free-parameter values [n][K] of design members member_offset .. member_offset + n - 1 (``sb`` a
    ``_cabi.SimplypSobol``)."""
    out = np.zeros((n, sb.n_free))
    load().sobol_host_design(C.byref(sb), C.c_int64(member_offset), C.c_int64(n), _ptr(out))
    return out


def picks(seed, n_boot, n):
    """Bootstrap positions [n_boot][n] (int64) of the resamples 0 .. n_boot - 1 over n used samples."""
    out = np.zeros((n_boot, n), dtype=np.uint32)
    for t in range(n_boot):
        load().sobol_host_picks(C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF), C.c_uint32(t), C.c_uint32(n),
                                C.c_int64(n), _ptr(out[t]))
    return out.astype(np.int64)
