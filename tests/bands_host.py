"""Test-only host build of the posterior predictive bands' arithmetic (simplyp_bands.cuh, see bands_host.cpp).

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
SRC = os.path.join(HERE, "bands_host.cpp")

_lib = None


def load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="simplyp_bands_host_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsimplyp_bands_host.so")
        # -ffp-contract=off: the host build must not fuse what the device forms with explicit roundings
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _i32(a, n):
    return np.ascontiguousarray(np.broadcast_to(np.asarray(a, dtype=np.int32), (n,)))


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def words(seed, member, day, series):
    """Philox words [n][4] (uint32) of the error draws of (member, day, series) (broadcast to one length)."""
    n = int(np.broadcast(np.asarray(member), np.asarray(day), np.asarray(series)).size)
    m, d, s = _i32(member, n), _i32(day, n), _i32(series, n)
    out = np.zeros((n, 4), dtype=np.uint32)
    load().bands_host_words(C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF), _ptr(m), _ptr(d), _ptr(s), _ptr(out),
                            C.c_int(n))
    return out


def epsilon(seed, member, day, series):
    """Standard normal deviates [n] of the error draws of (member, day, series)."""
    n = int(np.broadcast(np.asarray(member), np.asarray(day), np.asarray(series)).size)
    m, d, s = _i32(member, n), _i32(day, n), _i32(series, n)
    out = np.zeros(n)
    load().bands_host_epsilon(C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF), _ptr(m), _ptr(d), _ptr(s), _ptr(out),
                              C.c_int(n))
    return out


def nanquantile(x, q):
    """np.nanquantile(x, q, axis=-1) of x [R][N] through the host build of the index / interpolation functions,
    applied to NumPy-sorted rows: [n_q][R]."""
    x = np.atleast_2d(np.asarray(x, dtype=np.float64))
    R, N = x.shape
    srt = np.ascontiguousarray(np.sort(x, axis=-1))          # NaN last
    n = np.ascontiguousarray(np.sum(~np.isnan(x), axis=-1).astype(np.int64))
    q = np.ascontiguousarray(np.atleast_1d(np.asarray(q, dtype=np.float64)))
    out = np.zeros((q.size, R))
    if N > 0:
        load().bands_host_quantiles(_ptr(srt), _ptr(n), C.c_int64(R), C.c_int64(N), _ptr(q), C.c_int(q.size),
                                    _ptr(out))
    else:
        out[:] = np.nan
    return out


def keys(x):
    """(keys [n] uint64, values back from the keys [n])."""
    x = np.ascontiguousarray(np.asarray(x, dtype=np.float64).reshape(-1))
    k = np.zeros(x.size, dtype=np.uint64)
    back = np.zeros(x.size)
    load().bands_host_keys(_ptr(x), _ptr(k), _ptr(back), C.c_int64(x.size))
    return k, back
