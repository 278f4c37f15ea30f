"""TEST ONLY: ctypes binding of the per-problem-weight entry points of the CPU warp emulation (emu_weights_driver.cpp, which
compiles emu_driver.cpp and adds the PW = 1 instantiations of the kernel sources).  KCfg and kcfg_from_oracle come from emu.py."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu import KCfg, _HERE, _ROOT, _SRCS as _EMU_SRCS

_LIB = os.path.join(_HERE, "libmpc_emu_weights.so")
_SRCS = [os.path.join(_HERE, "emu_weights_driver.cpp")] + _EMU_SRCS


def build():
    if (not os.path.exists(_LIB)) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in _SRCS):
        subprocess.check_call(["/usr/bin/g++", "-O1", "-g", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-DMPC_HOST_EMU",
                               "-I" + _HERE, "-I" + os.path.join(_ROOT, "mkz_mpc_path_follower_b200", "csrc"),
                               "-x", "c++", _SRCS[0], "-o", _LIB])
    return _LIB


def _solve_w(fn_name, kcfg, state, ref, v_des, u_prev, w, warm, want_traj, tpp, slots):
    lib = C.CDLL(build())
    assert lib.emu_kcfg_size() == C.sizeof(KCfg)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    N = kcfg.N
    state = np.ascontiguousarray(state, dtype=np.float64); ref = np.ascontiguousarray(ref, dtype=np.float64)
    u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
    v_des = None if v_des is None else np.ascontiguousarray(v_des, dtype=np.float64)
    w = None if w is None else np.ascontiguousarray(w, dtype=np.float64)
    B = state.shape[0]
    p = lambda a: None if a is None else a.ctypes.data_as(dp)
    u0 = np.empty((B, 2)); cost = np.empty(B); status = np.empty(B, dtype=np.int32); iters = np.empty(B, dtype=np.int32)
    resto = np.empty(B, dtype=np.int32)
    traj = np.empty((B, 6 * N + 4)) if want_traj else None
    fn = getattr(lib, fn_name)
    args = [C.byref(kcfg), B, p(state), p(ref), p(v_des), p(u_prev), p(warm), p(w), p(u0), p(cost),
            status.ctypes.data_as(ip), iters.ctypes.data_as(ip), p(traj), resto.ctypes.data_as(ip)]
    types = [C.POINTER(KCfg), C.c_long] + [dp] * 8 + [ip, ip, dp, ip]
    if tpp:
        args.append(slots); types.append(C.c_long)
    fn.argtypes = types
    assert fn(*args) == 0
    return {"u0": u0, "cost": cost, "status": status, "iters": iters, "traj": traj, "n_resto": resto}


def solve_batch_w(kcfg, state, ref, v_des, u_prev, w, warm=None, want_traj=False, tpp=False, slots=3):
    """Per-problem cost weights w (B,8) (or None: kcfg.w through the per-problem path) on the emulated PW = 1 kernel source;
    tpp: the thread-per-problem solver.  A row that is negative or NaN gives that problem status 4 (ERROR), as with device pointers."""
    return _solve_w("emu_solve_batch_tpp_w" if tpp else "emu_solve_batch_w", kcfg, state, ref, v_des, u_prev, w, warm, want_traj, tpp, slots)


def solve_batch_frenet_w(kcfg, state, kpoly, v_des, u_prev, w, warm=None, want_traj=False, tpp=False, slots=3):
    """Frenet-frame variant with per-problem weights w (B,7) in set_cost_frenet's order."""
    return _solve_w("emu_solve_batch_tpp_frenet_w" if tpp else "emu_solve_batch_frenet_w", kcfg, state, kpoly, v_des, u_prev, w, warm,
                    want_traj, tpp, slots)


def rollout_w(kcfg, traj_table, pose0, T, w, track_using_time=True, target_vel=1.0, warm0=None, tpp=False):
    """rollout() with per-vehicle cost weights w (B,8) (mpcb200_rollout_w): the fused kernel's source, or tpp: the per-period pipeline."""
    lib = C.CDLL(build())
    dp = C.POINTER(C.c_double)
    pose0 = np.ascontiguousarray(np.atleast_2d(pose0), dtype=np.float64)
    B = pose0.shape[0]
    w = np.ascontiguousarray(w, dtype=np.float64)
    cols = [np.ascontiguousarray(traj_table[:, i]) for i in (0, 4, 5, 3, 6)]
    path_of = np.zeros(B, dtype=np.int32)
    log = np.zeros((T, B, 8)); final = np.zeros((B, 8))
    lib.emu_rollout_w.argtypes = [C.POINTER(KCfg), C.c_long, C.c_int, dp, C.POINTER(C.c_int), C.c_int, dp, dp, dp, dp, dp,
                                  C.c_int, C.c_double, dp, dp, dp, dp, C.c_int]
    w0 = None if warm0 is None else np.ascontiguousarray(warm0, dtype=np.float64)
    lib.emu_rollout_w(C.byref(kcfg), B, T, pose0.ctypes.data_as(dp), path_of.ctypes.data_as(C.POINTER(C.c_int)), traj_table.shape[0],
                      *[c.ctypes.data_as(dp) for c in cols], int(track_using_time), float(target_vel), w.ctypes.data_as(dp),
                      log.ctypes.data_as(dp), final.ctypes.data_as(dp), None if w0 is None else w0.ctypes.data_as(dp), int(bool(tpp)))
    return log, final
