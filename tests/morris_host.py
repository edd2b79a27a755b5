"""Test-only host build of the Morris screening's trajectory, design, selection and bootstrap arithmetic
(simplyp_morris.cuh, see morris_host.cpp).

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
SRC = os.path.join(HERE, "morris_host.cpp")

_lib = None


def load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="simplyp_morris_host_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsimplyp_morris_host.so")
        # -ffp-contract=off: the host build must not fuse what the device forms with explicit roundings
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _u64(seed):
    return C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF)


def levels(seed, K, p, n, c0=0):
    """Levels [n][K + 1][K] of candidates c0 .. c0 + n - 1."""
    out = np.zeros((n, K + 1, K), dtype=np.int32)
    load().morris_host_levels(_u64(seed), C.c_int64(c0), C.c_int64(n), C.c_int(K), C.c_int(p), _ptr(out))
    return out


def design(mo, member_offset, n, selected=None):
    """Free-parameter values [n][K] of design members member_offset .. member_offset + n - 1 (``mo`` a
    ``_cabi.SimplypMorris``)."""
    out = np.zeros((n, mo.n_free))
    sel = None if selected is None else np.ascontiguousarray(selected, dtype=np.int32)
    load().morris_host_design(C.byref(mo), None if sel is None else _ptr(sel), C.c_int64(member_offset),
                              C.c_int64(n), _ptr(out))
    return out


def select(mo):
    """Selected candidate indices [r] of ``mo``'s candidate pool."""
    out = np.zeros(mo.n_trajectories, dtype=np.int32)
    load().morris_host_select(C.byref(mo), _ptr(out))
    return out


def picks(seed, n_boot, n):
    """Bootstrap positions [n_boot][n] (int64) of the resamples 0 .. n_boot - 1 over n used trajectories."""
    out = np.zeros((n_boot, n), dtype=np.uint32)
    for b in range(n_boot):
        load().morris_host_picks(_u64(seed), C.c_uint32(b), C.c_uint32(n), C.c_int64(n), _ptr(out[b]))
    return out.astype(np.int64)
