"""ctypes binding of oracle/libmpc_oracle.so -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module.  PARITY UNPINNED: see oracle/mpc_oracle.h.
"""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libmpc_oracle.so")

STATUS_NAMES = {0: "Optimal", 1: "Infeasible", 2: "Unbounded", 3: "UserLimit", 4: "Error"}


class Cfg(C.Structure):
    _fields_ = [("N", C.c_int), ("dt", C.c_double), ("dt_control", C.c_double),
                ("L_a", C.c_double), ("L_b", C.c_double), ("v_min", C.c_double),
                ("v_max", C.c_double), ("a_max", C.c_double), ("steer_max", C.c_double),
                ("a_dmax", C.c_double), ("steer_dmax", C.c_double), ("w", C.c_double * 8),
                ("tol", C.c_double), ("max_iter", C.c_int),
                ("model", C.c_int), ("kpoly", C.c_double * 4)]


class Diag(C.Structure):
    _fields_ = [("dual_inf", C.c_double), ("constr_viol", C.c_double), ("compl_inf", C.c_double),
                ("mu_final", C.c_double), ("obj_scale", C.c_double), ("n_inertia_corr", C.c_int),
                ("n_soc", C.c_int), ("n_backtrack", C.c_int), ("ipopt_status", C.c_int), ("n_resto", C.c_int)]


class Path(C.Structure):
    _fields_ = [("n", C.c_int), ("t", C.POINTER(C.c_double)), ("X", C.POINTER(C.c_double)),
                ("Y", C.POINTER(C.c_double)), ("psi", C.POINTER(C.c_double)), ("s", C.POINTER(C.c_double))]


def build(force=False):
    src = os.path.join(_HERE, "mpc_oracle.c")
    if force or not os.path.exists(_LIB) or os.path.getmtime(_LIB) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            build()
        _lib = C.CDLL(_LIB)
        dp = C.POINTER(C.c_double)
        ip = C.POINTER(C.c_int)
        _lib.mpc_oracle_default_cfg.argtypes = [C.POINTER(Cfg), C.c_int]
        _lib.mpc_oracle_solve.argtypes = [C.POINTER(Cfg), dp, dp, C.c_double, dp, dp, dp, dp, dp, ip, ip, C.POINTER(Diag)]
        _lib.mpc_oracle_solve_batch.argtypes = [C.POINTER(Cfg), C.c_long, dp, dp, dp, dp, dp, dp, dp, ip, ip, dp, C.c_int]
        _lib.mpc_oracle_default_cfg_frenet.argtypes = [C.POINTER(Cfg), C.c_int]
        _lib.mpc_oracle_solve_batch_frenet.argtypes = [C.POINTER(Cfg), C.c_long, dp, dp, dp, dp, dp, dp, dp, ip, ip, dp, C.c_int]
        _lib.mpc_oracle_rollout_start.argtypes = [C.POINTER(Cfg), dp, dp, dp]
        _lib.mpc_oracle_eval_f.restype = C.c_double
        _lib.mpc_oracle_eval_f.argtypes = [C.POINTER(Cfg), dp, C.c_double, dp]
        _lib.mpc_oracle_eval_grad_f.argtypes = [C.POINTER(Cfg), dp, C.c_double, dp, dp]
        _lib.mpc_oracle_eval_c.argtypes = [C.POINTER(Cfg), dp, dp, dp]
        _lib.mpc_oracle_eval_d.argtypes = [C.POINTER(Cfg), dp, dp, dp]
        _lib.mpc_oracle_eval_jac.argtypes = [C.POINTER(Cfg), dp, dp, dp]
        _lib.mpc_oracle_eval_hess.argtypes = [C.POINTER(Cfg), dp, C.c_double, dp, dp]
        _lib.mpc_oracle_traj_to_z.argtypes = [C.POINTER(Cfg), dp, dp]
        _lib.mpc_oracle_z_to_traj.argtypes = [C.POINTER(Cfg), dp, dp]
        _lib.mpc_oracle_get_waypoints.argtypes = [C.POINTER(Path), C.c_int, C.c_double, C.c_double, C.c_double,
                                                  C.c_double, C.c_int, C.c_double, dp]
        _lib.mpc_oracle_plant_step.argtypes = [dp, C.c_double, C.c_double]
        _lib.mpc_oracle_closed_loop.argtypes = [C.POINTER(Cfg), C.POINTER(Path), dp, C.c_int, C.c_int,
                                                C.c_double, C.c_int, dp]
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _pi(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def default_cfg(N=8, weights=None, tol=None, max_iter=None, **kw):
    c = Cfg()
    lib().mpc_oracle_default_cfg(C.byref(c), N)
    if weights is not None:
        for i, v in enumerate(weights):
            c.w[i] = float(v)
    if tol is not None:
        c.tol = tol
    if max_iter is not None:
        c.max_iter = max_iter
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def solve(cfg, state, ref, v_des, u_prev, warm=None):
    """One solve.  ref: (3, N+1).  Returns dict."""
    N = cfg.N
    state = np.ascontiguousarray(state, dtype=np.float64)
    ref = np.ascontiguousarray(ref, dtype=np.float64).reshape(3 * (N + 1))
    u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
    warm = None if warm is None else np.ascontiguousarray(warm, dtype=np.float64)
    traj = np.empty(6 * N + 4)
    u0 = np.empty(2)
    cost = C.c_double()
    st = C.c_int()
    it = C.c_int()
    dg = Diag()
    rc = lib().mpc_oracle_solve(C.byref(cfg), _p(state), _p(ref), float(v_des), _p(u_prev), _p(warm), _p(traj), _p(u0),
                                C.byref(cost), C.byref(st), C.byref(it), C.byref(dg))
    assert rc == 0
    return {"traj": traj, "u0": u0, "cost": cost.value, "status": st.value, "iters": it.value,
            "diag": {f[0]: getattr(dg, f[0]) for f in Diag._fields_}}


def solve_batch(cfg, state, ref, v_des, u_prev, warm=None, want_traj=False, n_threads=1):
    N = cfg.N
    B = state.shape[0]
    state = np.ascontiguousarray(state, dtype=np.float64)
    ref = np.ascontiguousarray(ref, dtype=np.float64)
    u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
    v_des = None if v_des is None else np.ascontiguousarray(v_des, dtype=np.float64)
    u0 = np.empty((B, 2))
    cost = np.empty(B)
    status = np.empty(B, dtype=np.int32)
    iters = np.empty(B, dtype=np.int32)
    traj = np.empty((B, 6 * N + 4)) if want_traj else None
    n_resto = np.zeros(B, dtype=np.int32)
    L = lib()
    L.mpc_oracle_solve_batch_resto.argtypes = [C.POINTER(Cfg), C.c_long] + [C.c_void_p] * 11 + [C.c_int]
    rc = L.mpc_oracle_solve_batch_resto(C.byref(cfg), B, state.ctypes.data, ref.ctypes.data, None if v_des is None else v_des.ctypes.data,
                                        u_prev.ctypes.data, None if warm is None else warm.ctypes.data, u0.ctypes.data, cost.ctypes.data,
                                        status.ctypes.data, iters.ctypes.data, None if traj is None else traj.ctypes.data,
                                        n_resto.ctypes.data, int(n_threads))
    assert rc == 0
    return {"u0": u0, "cost": cost, "status": status, "iters": iters, "traj": traj, "n_resto": n_resto}


def default_cfg_frenet(N=8, weights=None, tol=None, max_iter=None, **kw):
    """MKZMPCPathFollowerFrenet.jl defaults; weights in the XY slot order (0, C_ey, C_epsi, C_ev, C_dacc, C_ddf, C_acc, C_df)."""
    c = Cfg()
    lib().mpc_oracle_default_cfg_frenet(C.byref(c), N)
    if weights is not None:
        for i, v in enumerate(weights):
            c.w[i] = float(v)
    if tol is not None:
        c.tol = tol
    if max_iter is not None:
        c.max_iter = max_iter
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def solve_batch_frenet(cfg, state, kpoly, v_des, u_prev, warm=None, want_traj=False, n_threads=1):
    """Frenet variant: state (B,4) = s, ey, epsi, v; kpoly (B,4) highest degree first."""
    N = cfg.N
    B = state.shape[0]
    state = np.ascontiguousarray(state, dtype=np.float64)
    kpoly = np.ascontiguousarray(kpoly, dtype=np.float64)
    assert kpoly.shape == (B, 4)
    u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
    v_des = None if v_des is None else np.ascontiguousarray(v_des, dtype=np.float64)
    u0 = np.empty((B, 2)); cost = np.empty(B)
    status = np.empty(B, dtype=np.int32); iters = np.empty(B, dtype=np.int32)
    traj = np.empty((B, 6 * N + 4)) if want_traj else None
    rc = lib().mpc_oracle_solve_batch_frenet(C.byref(cfg), B, _p(state), _p(kpoly), _p(v_des), _p(u_prev), _p(warm), _p(u0),
                                             _p(cost), _pi(status), _pi(iters), _p(traj), int(n_threads))
    assert rc == 0
    return {"u0": u0, "cost": cost, "status": status, "iters": iters, "traj": traj}


def module_load_solution(cfg):
    """Solution (traj order) of the module-load solve of the default problem (MKZMPCPathFollower.jl:126-128): the start
    point of the node's first solve."""
    t = np.zeros(6 * cfg.N + 4)
    lib().mpc_oracle_module_load_solution.argtypes = [C.POINTER(Cfg), C.POINTER(C.c_double)]
    lib().mpc_oracle_module_load_solution(C.byref(cfg), _p(t))
    return t


def rollout_start(cfg, state, u_prev):
    """Start points of MPCB200_START_ROLLOUT for a batch: (B, 6N+4) in traj order."""
    state = np.ascontiguousarray(state, dtype=np.float64); u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
    out = np.empty((state.shape[0], 6 * cfg.N + 4))
    for j in range(state.shape[0]):
        assert lib().mpc_oracle_rollout_start(C.byref(cfg), _p(state[j]), _p(u_prev[j]), _p(out[j])) == 0
    return out


def make_path(traj_table):
    """traj_table: the (n,7) table of GPSRefTrajectory.trajectory.  Returns (Path, keepalive)."""
    cols = [np.ascontiguousarray(traj_table[:, i]) for i in (0, 4, 5, 3, 6)]
    p = Path(traj_table.shape[0], *[_p(c) for c in cols])
    return p, cols


def get_waypoints(path, horizon, traj_dt, X, Y, yaw, v_target=None):
    ref = np.empty(3 * (horizon + 1))
    stop = lib().mpc_oracle_get_waypoints(C.byref(path), horizon, traj_dt, X, Y, yaw,
                                          0 if v_target is None else 1, 0.0 if v_target is None else v_target, _p(ref))
    return ref.reshape(3, horizon + 1), bool(stop)


def plant_step(st, acc_des, df_des):
    st = np.ascontiguousarray(st, dtype=np.float64).copy()
    lib().mpc_oracle_plant_step(_p(st), acc_des, df_des)
    return st


def closed_loop(cfg, path, pose0, T, track_using_time=True, target_vel=1.0, warm_start=True):
    log = np.zeros((T, 8))
    pose0 = np.ascontiguousarray(pose0, dtype=np.float64)
    n = lib().mpc_oracle_closed_loop(C.byref(cfg), C.byref(path), _p(pose0), T, int(track_using_time),
                                     float(target_vel), int(warm_start), _p(log))
    return log[:n]


def frenet_fit(xw, yw, window):
    """The reference of the Frenet node from the path ahead, as nav_msgs_path_frenet.py:44-86 computes it: xw, yw sampled on
    arange(0, window, 0.5) -> cubics X(s), Y(s) by np.polyfit (:65-70), their curvature on arange(0, window, 0.25) fitted by a
    cubic (:44-58), psi_start = atan2(Y'(0), X'(0)) (:84).  Returns (K_coeffs[4] highest degree first, psi_start)."""
    s_fit = np.arange(0.0, window, 0.5)
    s_interp = np.arange(0.0, window, 0.25)
    x_coeffs = np.polyfit(s_fit, xw, 3)
    y_coeffs = np.polyfit(s_fit, yw, 3)
    dx, dy = np.polyval(np.polyder(x_coeffs), s_interp), np.polyval(np.polyder(y_coeffs), s_interp)
    ddx, ddy = np.polyval(np.polyder(x_coeffs, 2), s_interp), np.polyval(np.polyder(y_coeffs, 2), s_interp)
    K = np.polyfit(s_interp, (dx * ddy - dy * ddx) / (dx * dx + dy * dy), 3)
    psi_start = float(np.arctan2(np.polyval(np.polyder(y_coeffs), 0.0), np.polyval(np.polyder(x_coeffs), 0.0)))
    return K, psi_start


def closed_loop_frenet(cfg, traj_table, pose0, T, window, target_vel, ey_from_path=True):
    """Closed loop on the Frenet-frame module (gazebo_sim_mpc_cmd_pub_frenet.jl:112-153) around the plant, one vehicle, with
    nothing from the library: per control period the plant (plant_step) runs ten publishes, the path ahead is the next `window`
    metres from the nearest sample (np.argmin, np.interp every 0.5 m, seen from the vehicle), frenet_fit gives K(s) and
    psi_start, and solve_batch_frenet solves from (0, e_y, -psi_start, v) with the previous solution as its start (all zeros in
    the first period) and cfg.max_iter as the cap.  e_y is the vehicle's offset from the fitted path start (ey_from_path) or 0.
    traj_table: the (n,7) table of GPSRefTrajectory.trajectory.  Returns the (T, 8) log of the rollouts:
    x, y, psi, v, acc_cmd, df_cmd, status, iters."""
    N = cfg.N
    Xp, Yp, sp = (np.ascontiguousarray(traj_table[:, i], dtype=np.float64) for i in (4, 5, 6))
    s_fit = np.arange(0.0, window, 0.5)
    st = np.array([pose0[0], pose0[1], pose0[2], 0.0, 0.0, 0.0, 0.0, 0.0])
    acc_des = df_des = 0.0
    u_prev = np.zeros((1, 2)); warm = np.zeros((1, 6 * N + 4)); log = np.zeros((T, 8))
    for t in range(T):
        for _ in range(10):
            st = plant_step(st, acc_des, df_des)
        i = int(np.argmin((Xp - st[0]) ** 2 + (Yp - st[1]) ** 2))
        sq = sp[i] + s_fit
        dx = np.interp(sq, sp, Xp) - st[0]; dy = np.interp(sq, sp, Yp) - st[1]
        c, s = np.cos(st[2]), np.sin(st[2])
        xw = c * dx + s * dy; yw = -s * dx + c * dy
        K, psi_start = frenet_fit(xw, yw, window)
        ey = -(-np.sin(psi_start) * xw[0] + np.cos(psi_start) * yw[0]) if ey_from_path else 0.0
        state = np.array([[0.0, ey, -psi_start, st[3]]])
        o = solve_batch_frenet(cfg, state, K[None], np.array([float(target_vel)]), u_prev, warm=warm)
        acc_des, df_des = float(o["u0"][0, 0]), float(o["u0"][0, 1])
        u_prev[0] = (df_des, acc_des)               # update_current_input(df_opt, a_opt) (:145)
        log[t] = (st[0], st[1], st[2], st[3], acc_des, df_des, o["status"][0], o["iters"][0])
    return log
