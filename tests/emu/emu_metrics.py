"""TEST ONLY: ctypes binding of the closed loops with tracking metrics on the CPU warp emulation (emu_metrics_driver.cpp, which
compiles emu_weights_driver.cpp and emu_driver.cpp and adds the MET = 1 instantiations of the kernel sources)."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu import KCfg, _HERE, _ROOT
from emu_weights import _SRCS as _W_SRCS

_LIB = os.path.join(_HERE, "libmpc_emu_metrics.so")
_SRCS = [os.path.join(_HERE, "emu_metrics_driver.cpp")] + _W_SRCS


def build():
    if (not os.path.exists(_LIB)) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in _SRCS):
        subprocess.check_call(["/usr/bin/g++", "-O1", "-g", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-DMPC_HOST_EMU",
                               "-I" + _HERE, "-I" + os.path.join(_ROOT, "mkz_mpc_path_follower_b200", "csrc"),
                               "-x", "c++", _SRCS[0], "-o", _LIB])
    return _LIB


def _cols(traj_table):
    return [np.ascontiguousarray(traj_table[:, i]) for i in (0, 4, 5, 3, 6)]


def rollout_metrics(kcfg, traj_table, pose0, T, w=None, pw=False, track_using_time=True, target_vel=1.0, warm0=None, tpp=False):
    """The XY closed loop with tracking metrics: the fused kernel's source (rollout_group<W, PW, 1>; pw selects PW = 1, w (B,8) or
    None = kcfg.w) or, tpp, the per-period pipeline with the metrics kernel's source.  Returns log (T,B,8), final (B,8), metrics (B,12)."""
    lib = C.CDLL(build())
    dp = C.POINTER(C.c_double)
    pose0 = np.ascontiguousarray(np.atleast_2d(pose0), dtype=np.float64)
    B = pose0.shape[0]
    w = None if w is None else np.ascontiguousarray(w, dtype=np.float64)
    path_of = np.zeros(B, dtype=np.int32)
    log = np.zeros((T, B, 8)); final = np.zeros((B, 8)); met = np.full((B, 12), -7.0)
    lib.emu_rollout_metrics.argtypes = [C.POINTER(KCfg), C.c_long, C.c_int, dp, C.POINTER(C.c_int), C.c_int, dp, dp, dp, dp, dp,
                                        C.c_int, C.c_double, dp, C.c_int, dp, dp, dp, C.c_int, dp]
    w0 = None if warm0 is None else np.ascontiguousarray(warm0, dtype=np.float64)
    p = lambda a: None if a is None else a.ctypes.data_as(dp)
    assert lib.emu_rollout_metrics(C.byref(kcfg), B, T, p(pose0), path_of.ctypes.data_as(C.POINTER(C.c_int)), traj_table.shape[0],
                                   *[p(c) for c in _cols(traj_table)], int(track_using_time), float(target_vel), p(w), int(bool(pw)),
                                   p(log), p(final), p(w0), int(bool(tpp)), p(met)) == 0
    return log, final, met


def rollout_frenet_metrics(kcfg, traj_table, pose0, T, window=40.0, target_vel=8.0, ey_from_path=True):
    """The fused Frenet closed loop with tracking metrics (rollout_group_frenet<1>).  Returns log (T,B,8), final (B,8), metrics (B,12)."""
    lib = C.CDLL(build())
    dp = C.POINTER(C.c_double)
    pose0 = np.ascontiguousarray(np.atleast_2d(pose0), dtype=np.float64)
    B = pose0.shape[0]
    path_of = np.zeros(B, dtype=np.int32)
    log = np.zeros((T, B, 8)); final = np.zeros((B, 8)); met = np.full((B, 12), -7.0)
    lib.emu_rollout_frenet_metrics.argtypes = [C.POINTER(KCfg), C.c_long, C.c_int, dp, C.POINTER(C.c_int), C.c_int, dp, dp, dp, dp, dp,
                                               C.c_double, C.c_double, C.c_int, dp, dp, dp]
    p = lambda a: a.ctypes.data_as(dp)
    assert lib.emu_rollout_frenet_metrics(C.byref(kcfg), B, T, p(pose0), path_of.ctypes.data_as(C.POINTER(C.c_int)), traj_table.shape[0],
                                          *[p(c) for c in _cols(traj_table)], float(window), float(target_vel), int(bool(ey_from_path)),
                                          p(log), p(final), p(met)) == 0
    return log, final, met
