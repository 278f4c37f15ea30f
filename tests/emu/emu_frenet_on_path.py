"""TEST ONLY: ctypes binding of the reference pass of mpcb200_solve_batch_frenet_on_path on the CPU warp emulation
(emu_frenet_on_path_driver.cpp, which compiles emu_frenet_driver.cpp and adds frenet_on_path_problem on one warp per problem).
KCfg and kcfg_from_oracle come from emu.py; the solves of the returned rows are emu.solve_batch_frenet and
emu_weights.solve_batch_frenet_w."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu import KCfg, _HERE, _ROOT, _SRCS as _EMU_SRCS
from emu_frenet import Tables3, _tables

_LIB = os.path.join(_HERE, "libmpc_emu_frenet_on_path.so")
_SRCS = [os.path.join(_HERE, "emu_frenet_on_path_driver.cpp"), os.path.join(_HERE, "emu_frenet_driver.cpp")] + _EMU_SRCS
_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)


def build():
    if (not os.path.exists(_LIB)) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in _SRCS):
        subprocess.check_call(["/usr/bin/g++", "-O1", "-g", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-DMPC_HOST_EMU",
                               "-I" + _HERE, "-I" + os.path.join(_ROOT, "mkz_mpc_path_follower_b200", "csrc"),
                               "-x", "c++", _SRCS[0], "-o", _LIB])
    return _LIB


def frenet_on_path(kcfg, traj_tables, pose, path_of, window, ey_from_path=True, unset=()):
    """frenet_on_path_problem for B problems: pose (B,4) = X, Y, psi, v; path_of (B,) into the one to three (n,7) tables;
    `unset`: table ids handled as never set.  Returns k_coeffs (B,4), state (B,4) = (0, e_y, -psi_start, v)."""
    lib = C.CDLL(build())
    assert lib.emu_kcfg_size() == C.sizeof(KCfg)
    pose = np.ascontiguousarray(np.atleast_2d(pose), dtype=np.float64)
    B = pose.shape[0]
    path_of = np.ascontiguousarray(path_of, dtype=np.int32)
    assert pose.shape == (B, 4) and path_of.shape == (B,)
    tb, keep = _tables(traj_tables)
    k = np.full((B, 4), -1.0); st = np.full((B, 4), -1.0)
    lib.emu_frenet_on_path.argtypes = [C.POINTER(KCfg), C.POINTER(Tables3), C.c_int, C.c_double, C.c_int, C.c_long, _dp, _ip, _dp, _dp]
    assert lib.emu_frenet_on_path(C.byref(kcfg), C.byref(tb), sum(1 << i for i in unset), float(window), int(bool(ey_from_path)), B,
                                  pose.ctypes.data_as(_dp), path_of.ctypes.data_as(_ip), k.ctypes.data_as(_dp), st.ctypes.data_as(_dp)) == 0
    return k, st
