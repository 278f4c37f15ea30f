"""TEST ONLY: ctypes binding of the Frenet closed-loop hooks of the CPU warp emulation (emu_frenet_driver.cpp, which compiles
emu_driver.cpp and adds frenet_reference on one warp, the fit-matrix helpers, the fused loop over three path tables and the
per-period pipeline).  KCfg and kcfg_from_oracle come from emu.py."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu import KCfg, _HERE, _ROOT, _SRCS as _EMU_SRCS

_LIB = os.path.join(_HERE, "libmpc_emu_frenet.so")
_SRCS = [os.path.join(_HERE, "emu_frenet_driver.cpp")] + _EMU_SRCS
_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)


class Tables3(C.Structure):
    _fields_ = [("n", _ip), ("t", C.POINTER(_dp)), ("X", C.POINTER(_dp)), ("Y", C.POINTER(_dp)), ("psi", C.POINTER(_dp)),
                ("s", C.POINTER(_dp))]


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


def _tables(traj_tables):
    """Tables3 over one to three (n,7) tables of GPSRefTrajectory.trajectory (unused slots repeat the last); returns (struct, keepalive)."""
    traj_tables = list(traj_tables)
    assert 1 <= len(traj_tables) <= 3
    traj_tables += [traj_tables[-1]] * (3 - len(traj_tables))
    cols = [[np.ascontiguousarray(tb[:, i], dtype=np.float64) for tb in traj_tables] for i in (0, 4, 5, 3, 6)]
    n = np.array([tb.shape[0] for tb in traj_tables], dtype=np.int32)
    arrs = [(_dp * 3)(*[c.ctypes.data_as(_dp) for c in col]) for col in cols]
    return Tables3(n.ctypes.data_as(_ip), *arrs), (n, cols, arrs)


def fit_grid_sizes(window):
    """(n1, n2): the sizes of the fit grids the library builds for `window` (fit_grid_sizes in mpc_kernel.cuh)."""
    n1, n2 = C.c_int(), C.c_int()
    lib = _lib()
    lib.emu_fit_grid_sizes.argtypes = [C.c_double, _ip, _ip]
    lib.emu_fit_grid_sizes(float(window), C.byref(n1), C.byref(n2))
    return n1.value, n2.value


def cubic_fit_matrix(n, step):
    """The host-built (4, n) least-squares cubic fit matrix on the grid g * step, g < n (cubic_fit_matrix in mpc_kernel.cuh)."""
    P = np.empty((4, n))
    lib = _lib()
    lib.emu_cubic_fit_matrix.argtypes = [C.c_int, C.c_double, _dp]
    lib.emu_cubic_fit_matrix(int(n), float(step), P.ctypes.data_as(_dp))
    return P


def frenet_reference(kcfg, traj_table, poses, window, ey_from_path=True):
    """frenet_reference on one emulated warp for each (X, Y, yaw) of poses (M,3) on the path traj_table.  Returns dict with
    kc (M,4), ey (M,), psi0 (M,), and what the kernel samples: nearest (M,) sample index, xw, yw (M, n1) the path ahead every
    0.5 m in the vehicle frame."""
    lib = _lib()
    poses = np.ascontiguousarray(np.atleast_2d(poses), dtype=np.float64)
    M = poses.shape[0]
    n1, _ = fit_grid_sizes(window)
    tb, keep = _tables([traj_table])
    kc = np.empty((M, 4)); ey = np.empty(M); psi0 = np.empty(M); bi = np.empty(M, dtype=np.int32)
    xw = np.empty((M, n1)); yw = np.empty((M, n1))
    lib.emu_frenet_reference.argtypes = [C.POINTER(KCfg), C.POINTER(Tables3), C.c_double, C.c_int, C.c_long, _dp, _dp, _dp, _dp, _ip, _dp, _dp]
    assert lib.emu_frenet_reference(C.byref(kcfg), C.byref(tb), float(window), int(bool(ey_from_path)), M, poses.ctypes.data_as(_dp),
                                    kc.ctypes.data_as(_dp), ey.ctypes.data_as(_dp), psi0.ctypes.data_as(_dp), bi.ctypes.data_as(_ip),
                                    xw.ctypes.data_as(_dp), yw.ctypes.data_as(_dp)) == 0
    return {"kc": kc, "ey": ey, "psi0": psi0, "nearest": bi, "xw": xw, "yw": yw}


def rollout_frenet3(kcfg, traj_tables, pose0, path_of, T, window=40.0, target_vel=8.0, ey_from_path=True, tpp=False):
    """mpcb200_rollout_frenet on the emulator with up to three path tables: vehicle v on traj_tables[path_of[v]].  The fused
    kernel's source (rollout_group_frenet), or tpp: the per-period pipeline.  Returns log (T,B,8), final (B,8)."""
    lib = _lib()
    pose0 = np.ascontiguousarray(np.atleast_2d(pose0), dtype=np.float64)
    B = pose0.shape[0]
    path_of = np.ascontiguousarray(path_of, dtype=np.int32)
    assert path_of.shape == (B,) and (path_of >= 0).all() and (path_of < len(traj_tables)).all()
    tb, keep = _tables(traj_tables)
    log = np.zeros((T, B, 8)); final = np.zeros((B, 8))
    fn = lib.emu_rollout_frenet_tpp if tpp else lib.emu_rollout_frenet3
    fn.argtypes = [C.POINTER(KCfg), C.c_long, C.c_int, _dp, _ip, C.POINTER(Tables3), C.c_double, C.c_double, C.c_int, _dp, _dp]
    assert fn(C.byref(kcfg), B, int(T), pose0.ctypes.data_as(_dp), path_of.ctypes.data_as(_ip), C.byref(tb), float(window),
              float(target_vel), int(bool(ey_from_path)), log.ctypes.data_as(_dp), final.ctypes.data_as(_dp)) == 0
    return log, final
