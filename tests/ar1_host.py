"""Test-only host build of the AR(1) error model's arithmetic and of the sampler's parameter-row writes (see
ar1_host.cpp).

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
SRC = os.path.join(HERE, "ar1_host.cpp")

_lib = None


def load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="simplyp_ar1_host_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsimplyp_ar1_host.so")
        # -ffp-contract=off: the host build must not fuse what the device forms with explicit roundings
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, SRC])
        _lib = C.CDLL(so)
        _lib.ar1_host_row.restype = C.c_double
        _lib.ar1_host_row.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_double]
    return _lib


def row(o, s, m, phi):
    """LOGLIK of one series (observations o [D], NaN where not observed; simulated values s [D]) as the kernel sums
    it."""
    o = np.ascontiguousarray(o, dtype=np.float64)
    s = np.ascontiguousarray(s, dtype=np.float64)
    assert o.shape == s.shape and o.ndim == 1
    return float(load().ar1_host_row(o.ctypes.data, s.ctypes.data, o.size, float(m), float(phi)))


def write_targets(params, n_sc, values, mrow, srow):
    """mcmc_write_target of every free parameter (``params``: a ctypes array of SimplypMcmcParam) into mrow [NP_MEMBER]
    and srow [S][NP_SC], in place."""
    values = np.ascontiguousarray(values, dtype=np.float64)
    for a in (mrow, srow):
        assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    load().ar1_host_write_targets(params, C.c_int(len(values)), C.c_int(int(n_sc)), values.ctypes.data_as(C.c_void_p),
                                  mrow.ctypes.data_as(C.c_void_p), srow.ctypes.data_as(C.c_void_p))
