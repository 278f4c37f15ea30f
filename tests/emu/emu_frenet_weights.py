"""TEST ONLY: ctypes binding of the Frenet closed loop with per-vehicle cost weights on the CPU warp emulation
(emu_frenet_weights_driver.cpp, which compiles emu_frenet_driver.cpp and emu_driver.cpp and adds the PW = 1 forms of the fused
loop and the per-period pipeline).  The library has its own copy of the emulator's race check: race_check / race_count here."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu import KCfg, _HERE, _ROOT
from emu_frenet import Tables3, _tables, _SRCS as _F_SRCS

_LIB = os.path.join(_HERE, "libmpc_emu_frenet_weights.so")
_SRCS = [os.path.join(_HERE, "emu_frenet_weights_driver.cpp")] + _F_SRCS
_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)


def build():
    if (not os.path.exists(_LIB)) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in _SRCS):
        subprocess.check_call(["/usr/bin/g++", "-O1", "-g", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-DMPC_HOST_EMU",
                               "-I" + _HERE, "-I" + os.path.join(_ROOT, "mkz_mpc_path_follower_b200", "csrc"),
                               "-x", "c++", _SRCS[0], "-o", _LIB])
    return _LIB


def _lib():
    lib = C.CDLL(build())
    assert lib.emu_kcfg_size() == C.sizeof(KCfg)
    return lib


def race_check(on=True):
    _lib().emu_race_enable(1 if on else 0)


def race_count():
    lib = _lib()
    lib.emu_race_count.restype = C.c_long
    return lib.emu_race_count()


def rollout_frenet_w(kcfg, traj_tables, pose0, path_of, T, w, window=40.0, target_vel=8.0, ey_from_path=True, metrics=False,
                     tpp=False):
    """mpcb200_rollout_frenet_w on the emulator: vehicle v on traj_tables[path_of[v]] with the cost weights w[v] (B,7) in every
    period.  The fused kernel's source (rollout_group_frenet<MET, 1>) or, tpp, the per-period pipeline (TppSolverT<1, 1>).
    Returns log (T,B,8), final (B,8) and, metrics (fused only), metrics (B,12)."""
    lib = _lib()
    pose0 = np.ascontiguousarray(np.atleast_2d(pose0), dtype=np.float64)
    B = pose0.shape[0]
    path_of = np.ascontiguousarray(path_of, dtype=np.int32)
    w = np.ascontiguousarray(w, dtype=np.float64)
    assert path_of.shape == (B,) and w.shape == (B, 7) and (path_of >= 0).all() and (path_of < len(traj_tables)).all()
    tb, keep = _tables(traj_tables)
    log = np.zeros((T, B, 8)); final = np.zeros((B, 8)); met = np.full((B, 12), -7.0) if metrics else None
    fn = lib.emu_rollout_frenet_w
    fn.argtypes = [C.POINTER(KCfg), C.c_long, C.c_int, _dp, _ip, C.POINTER(Tables3), C.c_double, C.c_double, C.c_int, _dp, _dp, _dp,
                   _dp, C.c_int]
    assert fn(C.byref(kcfg), B, int(T), pose0.ctypes.data_as(_dp), path_of.ctypes.data_as(_ip), C.byref(tb), float(window),
              float(target_vel), int(bool(ey_from_path)), w.ctypes.data_as(_dp), log.ctypes.data_as(_dp), final.ctypes.data_as(_dp),
              None if met is None else met.ctypes.data_as(_dp), int(bool(tpp))) == 0
    return (log, final, met) if metrics else (log, final)
