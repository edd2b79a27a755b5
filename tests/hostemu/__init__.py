"""Test-only host build of the kernels' per-thread arithmetic (see hostemu.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SRC = os.path.join(HERE, "hostemu.cpp")
LIB = os.path.join(HERE, "libsimplyp_hostemu.so")
DEPS = [SRC, os.path.join(ROOT, "simplyp_b200", "csrc", "simplyp_core.cuh"),
        os.path.join(HERE, "scalar_program.h"),
        os.path.join(ROOT, "simplyp_b200", "csrc", "simplyp_quad.cuh"),
        os.path.join(ROOT, "simplyp_b200", "csrc", "simplyp_plan.cuh"),
        os.path.join(ROOT, "include", "simplyp_b200.h")]

_lib = None


def build(force=False):
    stale = force or not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in DEPS)
    if stale:
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas",
                               "-o", LIB, SRC])
    return LIB


def load():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def run_quad(forcing, member_params, sc_params, parent_offsets, parent_ids, opt):
    """The quad program (4 lanes per member) executed by the host build (tests only)."""
    return run(forcing, member_params, sc_params, parent_offsets, parent_ids, opt, entry="hostemu_run_quad")


def run(forcing, member_params, sc_params, parent_offsets, parent_ids, opt, entry="hostemu_run"):
    """Same contract as simplyp_b200._cabi.run_host, executed by the host build (tests only)."""
    from simplyp_b200 import _cabi, packing as pk
    lib = load()
    forcing = np.ascontiguousarray(forcing, dtype=np.float64)
    member_params = np.ascontiguousarray(member_params, dtype=np.float64)
    sc_params = np.ascontiguousarray(sc_params, dtype=np.float64)
    if sc_params.ndim == 2:
        sc_params = sc_params[None]
    M, D = member_params.shape[0], forcing.shape[0]
    Msc, S = sc_params.shape[0], sc_params.shape[1]
    po = np.ascontiguousarray(parent_offsets, dtype=np.int32)
    pid = np.ascontiguousarray(parent_ids, dtype=np.int32)
    if pid.size == 0:
        pid = np.zeros(1, dtype=np.int32)
    dims = _cabi.make_dims(M, S, D, Msc, 0, int(po[-1]))
    out = np.zeros((M, S, D, pk.NOUT))
    diag = np.zeros((M, S, pk.NDIAG), dtype=np.int64)
    vp = C.c_void_p
    getattr(lib, entry)(C.byref(dims), C.byref(opt), forcing.ctypes.data_as(vp), member_params.ctypes.data_as(vp),
                    sc_params.ctypes.data_as(vp), po.ctypes.data_as(vp), pid.ctypes.data_as(vp),
                    out.ctypes.data_as(vp), diag.ctypes.data_as(vp))
    return out, diag


def quad_rhs_check(member_row, sc_row, P, E, doy, us, y7, dynamic_epc0=1, dynamic_erod=1):
    """Largest relative difference between the quad formulation's derivatives and rhs() at one state."""
    lib = load()
    lib.hostemu_quad_rhs_check.restype = C.c_double
    lib.hostemu_quad_rhs_check.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_void_p,
                                           C.c_void_p, C.c_int, C.c_int]
    mp = np.ascontiguousarray(member_row, dtype=np.float64)
    sp = np.ascontiguousarray(sc_row, dtype=np.float64)
    us = np.ascontiguousarray(us, dtype=np.float64)
    y7 = np.ascontiguousarray(y7, dtype=np.float64)
    return float(lib.hostemu_quad_rhs_check(mp.ctypes.data, sp.ctypes.data, P, E, doy, us.ctypes.data,
                                            y7.ctypes.data, dynamic_epc0, dynamic_erod))


def exp_tab(x):
    """sp_exp_tab of simplyp_core.cuh evaluated on the host."""
    lib = load()
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.empty_like(x)
    lib.hostemu_exp_tab(x.ctypes.data_as(C.c_void_p), y.ctypes.data_as(C.c_void_p), C.c_int(x.size))
    return y


def run_quad_split(forcing, member_params, sc_params, parent_offsets, parent_ids, opt, split):
    """The quad program over days [0, split) and then, continued from the stored midnight state, [split, D)."""
    from simplyp_b200 import _cabi, packing as pk
    lib = load()
    forcing = np.ascontiguousarray(forcing, dtype=np.float64)
    member_params = np.ascontiguousarray(member_params, dtype=np.float64)
    sc_params = np.ascontiguousarray(sc_params, dtype=np.float64)
    if sc_params.ndim == 2:
        sc_params = sc_params[None]
    M, D = member_params.shape[0], forcing.shape[0]
    po = np.ascontiguousarray(parent_offsets, dtype=np.int32)
    pid = np.zeros(1, dtype=np.int32)
    dims = _cabi.make_dims(M, 1, D, sc_params.shape[0], 0, 0)
    out = np.zeros((M, 1, D, pk.NOUT))
    diag = np.zeros((M, 1, pk.NDIAG), dtype=np.int64)
    vp = C.c_void_p
    rc = lib.hostemu_run_quad_split(C.byref(dims), C.byref(opt), forcing.ctypes.data_as(vp),
                                    member_params.ctypes.data_as(vp), sc_params.ctypes.data_as(vp),
                                    po.ctypes.data_as(vp), pid.ctypes.data_as(vp), out.ctypes.data_as(vp),
                                    diag.ctypes.data_as(vp), C.c_int(int(split)))
    assert rc == 0
    return out, diag


LAUNCH_CONFIG_FIELDS = ("grid", "minb", "pilot_days", "pilot_minb", "plan", "nY", "nP", "Q", "resident", "solo",
                        "epoch_days", "n_epochs")


def launch_config(M, D, n_sm, network=False, n_levels=0, grid_one_epoch=0, pilot_days=0, workspace=True):
    """launch_config() of simplyp_plan.cuh under the SIMPLYP_* overrides in os.environ, as a dict of
    LAUNCH_CONFIG_FIELDS."""
    lib = load()
    out = np.zeros(len(LAUNCH_CONFIG_FIELDS), dtype=np.int64)
    lib.hostemu_launch_config(C.c_int(M), C.c_int(D), C.c_int(int(network)), C.c_int(n_levels),
                              C.c_longlong(grid_one_epoch), C.c_int(pilot_days), C.c_int(int(workspace)), C.c_int(n_sm),
                              out.ctypes.data_as(C.c_void_p))
    return dict(zip(LAUNCH_CONFIG_FIELDS, (int(x) for x in out)))


def plan(M, n_sm, solo, resident=2):
    """Placement plan arithmetic: (index_of_rank [M], list_of_block [B], pos_in_list [B],
    (nY, nP, Q, n_lists, n_launch, resident)) or None."""
    lib = load()
    B = (M + 31) // 32
    idx = np.zeros(M, dtype=np.int32)
    lst = np.zeros(B, dtype=np.int32)
    pos = np.zeros(B, dtype=np.int32)
    shape = np.zeros(6, dtype=np.int32)
    vp = C.c_void_p
    rc = lib.hostemu_plan(C.c_int(M), C.c_int(n_sm), C.c_int(solo), C.c_int(resident), idx.ctypes.data_as(vp), lst.ctypes.data_as(vp),
                          pos.ctypes.data_as(vp), shape.ctypes.data_as(vp))
    assert rc >= 0, "a virtual block is out of range or sits in two lists"
    return None if rc == 0 else (idx, lst, pos, tuple(int(x) for x in shape))
