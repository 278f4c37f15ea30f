"""Closed-loop harness: the control step of scripts/mpc_cmd_pub.jl:86-157 driving the plant of
scripts/vehicle_simulator.py, for one vehicle (the reference workload, BASELINE.json configs[0]) or a
batch of independent vehicles (configs[3]).

Per 10 Hz control step, exactly as `pub_loop` does:
  1. latch the latest state_est (x, y, psi, v -- msg.a / msg.df are NOT used, :72-84)
  2. waypoints from GPSRefTrajectory.get_waypoints (time mode when track_using_time, :99-112);
     a stop_cmd latches command_stop for good
  3. update_init_cond / update_reference (:115-116)
  4. if not stopped: solve_model -> publish MPC_cmd (acc, steer) WHATEVER the status (:121-132),
     then update_current_input(df_opt, a_opt) (:140); the next solve starts from this solution
  5. if stopped: publish (-1.0, 0.0) (:148-153)
and the plant runs 10 publishes (100 Euler sub-steps) per control period.

This host-driven version calls libmpc_b200 once per control step for the whole batch
(mpcb200_solve_batch); the fully on-device loop is mpcb200_rollout.
"""
import numpy as np

from . import capi
from .gps_ref_traj import GPSRefTrajectory
from .vehicle_simulator import VehicleSimulator


def run(path_ids, pose0, T, N=8, dt=0.2, track_using_time=True, target_vel=1.0, solver=None, warm_start=True,
        weights=(9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0)):
    """path_ids: (B,) ints in 1..3; pose0: (B,3) X0, Y0, Psi0.  Returns dict with log (T,B,8) =
    x, y, psi, v, acc_cmd, df_cmd, status, iters (status -1 where the stop latch is set)."""
    path_ids = np.atleast_1d(np.asarray(path_ids)); pose0 = np.atleast_2d(np.asarray(pose0, dtype=np.float64))
    B = path_ids.shape[0]
    own = solver is None
    if own:
        solver = capi.Solver(N)
        solver.set_cost(weights)
    trajs = {p: GPSRefTrajectory(mat_filename=int(p), traj_horizon=N, traj_dt=dt) for p in sorted(set(path_ids.tolist()))}
    sim = VehicleSimulator(X0=pose0[:, 0], Y0=pose0[:, 1], Psi0=pose0[:, 2], batch=B)
    des_speed = target_vel if target_vel > 0.0 else 0.0          # mpc_cmd_pub.jl:58-62
    u_curr = np.zeros((B, 2))                                    # d_f_current, acc_current = 0 (:75,:82)
    # the first solve starts from the solution of the module-load solve of the default problem (MKZMPCPathFollower.jl:
    # 126-128; JuMP re-solves from the previous primal values), every later one from the previous solution
    warm = np.repeat(module_load_solution(N, device=solver.cfg.device)[None], B, axis=0)
    command_stop = np.zeros(B, dtype=bool)
    log = np.zeros((T, B, 8))
    ref = np.empty((B, 3, N + 1))
    for t in range(T):
        for _ in range(10):
            sim.update_vehicle_model()
        st = sim.state_est()[:, :4].copy()
        for p, g in trajs.items():
            m = path_ids == p
            r, stop = g.get_waypoints_batch(st[m, 0], st[m, 1], st[m, 2], v_target=None if track_using_time else des_speed)
            ref[m] = r
            command_stop[m] |= stop
        out = solver.solve_batch(st, ref, u_curr, v_des=np.full(B, des_speed), warm=warm if warm_start else None)
        act = ~command_stop
        acc = np.where(act, out["u0"][:, 0], -1.0)
        dfc = np.where(act, out["u0"][:, 1], 0.0)
        sim.mpc_cmd(acc, dfc)
        u_curr[act, 0] = out["u0"][act, 1]       # update_current_input(df_opt, a_opt): steering first
        u_curr[act, 1] = out["u0"][act, 0]
        log[t, :, 0:4] = st
        log[t, :, 4] = acc; log[t, :, 5] = dfc
        log[t, :, 6] = np.where(act, out["status"], -1); log[t, :, 7] = np.where(act, out["iters"], 0)
    if own:
        solver.close()
    return {"log": log, "final_state": sim.full_state(), "command_stop": command_stop}


_seed_cache = {}


def module_load_solution(N, device=0):
    """(6N+4,) solution of the default problem of MKZMPCPathFollower.jl:36-39,75,82,110-113 (zero state and previous
    command, x_ref = 15 t, y_ref = psi_ref = 0, v_target = 15, module-default weights, start = 0.0), solved by the library."""
    if N not in _seed_cache:
        s = capi.Solver(N, device=device)   # a fresh handle holds the module-default weights
        ref = np.zeros((1, 3, N + 1)); ref[0, 0] = 15.0 * (np.arange(N + 1) * s.cfg.dt)
        out = s.solve_batch(np.zeros((1, 4)), ref, np.zeros((1, 2)), v_des=np.array([15.0]), want_traj=True)
        s.close()
        _seed_cache[N] = out["traj"][0].copy()
    return _seed_cache[N]


def _nearest_samples(traj_table, xy):
    """Nearest path sample of each pose xy (M,2) over the whole path (np.argmin, first index on ties, as ref_gps_traj.py:136-137
    and TeamSolver::nearest_sample): (index (M,), squared distance (M,))."""
    XY = traj_table[:, 4:6]
    d = (XY[None, :, 0] - xy[:, 0:1]) ** 2 + (XY[None, :, 1] - xy[:, 1:2]) ** 2
    i = d.argmin(axis=1)
    return i, d[np.arange(d.shape[0]), i]


def path_errors(log, traj_table):
    """Tracking-quality metric of scripts/analysis/plot_path_tracking_error.py:21-34: distance to the
    nearest path sample for every logged pose.  log (T,B,8) -> (T,B)."""
    T, B = log.shape[0], log.shape[1]
    err = np.empty((T, B))
    for t in range(T):
        err[t] = np.sqrt(_nearest_samples(traj_table, log[t, :, 0:2])[1])
    return err


def tracking_metrics(log, traj_table):
    """Per-vehicle tracking metrics of a closed-loop log (T,B,8) on one path (the (n,7) table of GPSRefTrajectory.trajectory):
    (B,12) in the order of capi.ROLLOUT_METRICS, as mpcb200_rollout_metrics / _frenet_metrics accumulate them on the device
    (include/mpc_b200.h).  A period counts when a solve ran in it (status >= 0); e is the distance to the nearest path sample i of
    the logged pose, h = mod(psi - psi_i + pi, 2 pi) - pi, the command rates are against the previous counting period's commands
    (0 before the first).  The sums run in period order, so the device's results are reproduced to the last bit."""
    T, B = log.shape[0], log.shape[1]
    psi_p, s_p = traj_table[:, 3], traj_table[:, 6]
    n, se, se2, emax, sh2, hmax, sda2, sdd2, nno, it, pa, pd = (np.zeros(B) for _ in range(12))
    s_last = np.full(B, np.nan)
    stop = np.full(B, -1.0)
    for t in range(T):
        status = log[t, :, 6]
        stop[(status < 0) & (stop < 0)] = t
        c = status >= 0
        if not c.any():
            continue
        i, d = _nearest_samples(traj_table, log[t, c, 0:2])
        e = np.sqrt(d)
        h = np.mod(log[t, c, 2] - psi_p[i] + np.pi, 2.0 * np.pi) - np.pi
        acc, dfc = log[t, c, 4], log[t, c, 5]
        da, dd = acc - pa[c], dfc - pd[c]
        n[c] += 1.0
        se[c] += e
        se2[c] += e * e
        emax[c] = np.maximum(emax[c], e)
        sh2[c] += h * h
        hmax[c] = np.maximum(hmax[c], np.abs(h))
        sda2[c] += da * da
        sdd2[c] += dd * dd
        nno[c] += status[c] != 0
        it[c] += log[t, c, 7]
        s_last[c] = s_p[i]
        pa[c] = acc
        pd[c] = dfc
    out = np.zeros((B, 12))
    m = n > 0
    nm = n[m]
    out[:, 0] = n
    out[m, 1] = se[m] / nm
    out[m, 2] = np.sqrt(se2[m] / nm)
    out[m, 3] = emax[m]
    out[m, 4] = np.sqrt(sh2[m] / nm)
    out[m, 5] = hmax[m]
    out[m, 6] = np.sqrt(sda2[m] / nm)
    out[m, 7] = np.sqrt(sdd2[m] / nm)
    out[m, 8] = nno[m]
    out[m, 9] = it[m]
    out[:, 10] = s_last
    out[:, 11] = stop
    return out


def run_frenet(path_ids, pose0, T, N=8, window=40.0, target_vel=8.0, solver=None, ey_from_path=True):
    """Closed loop on the Frenet-frame module: the control step of
    scripts/nodes_gazebo_sim/gazebo_sim_mpc_cmd_pub_frenet.jl:112-153 around the plant of scripts/vehicle_simulator.py
    (Gazebo, which drives that node in the reference, is out of scope; this is the same loop on the repository's plant).

    Per 10 Hz step: the next `window` metres of the path from the sample nearest to the vehicle, in the vehicle frame
    (the node's `target_path` message, :90-119) -> K_coeffs, psi_start = get_reference_frenet (:100) ->
    update_init_cond(0, e_y, -psi_start, v) (:125), update_reference(path, K_coeffs, des_speed) (:126), solve_model
    (:130), publish the command whatever the status (:139-143), update_current_input(df_opt, a_opt) (:145); every solve
    starts from the previous solution.  The node passes e_y = 0 (it relies on a path that starts at the vehicle);
    ey_from_path = True (default) passes the vehicle's lateral offset from the fitted path start instead, which is
    what makes the loop hold the lane on a recorded path that does not start at the vehicle.
    Returns dict with log (T,B,8) = x, y, psi, v, acc_cmd, df_cmd, status, iters."""
    from . import frenet_ref
    path_ids = np.atleast_1d(np.asarray(path_ids)); pose0 = np.atleast_2d(np.asarray(pose0, dtype=np.float64))
    B = path_ids.shape[0]
    own = solver is None
    if own:
        solver = capi.FrenetSolver(N)
    tables = {p: GPSRefTrajectory(mat_filename=int(p), traj_horizon=N, traj_dt=0.2).trajectory for p in sorted(set(path_ids.tolist()))}
    sim = VehicleSimulator(X0=pose0[:, 0], Y0=pose0[:, 1], Psi0=pose0[:, 2], batch=B)
    u_curr = np.zeros((B, 2)); warm = np.zeros((B, 6 * N + 4))
    s_fit = np.arange(0.0, window, 0.5)
    log = np.zeros((T, B, 8))
    state = np.zeros((B, 4)); kpoly = np.zeros((B, 4))
    for t in range(T):
        for _ in range(10):
            sim.update_vehicle_model()
        st = sim.state_est()[:, :4].copy()
        xw = np.empty((B, s_fit.size)); yw = np.empty_like(xw)
        for b in range(B):
            tr = tables[int(path_ids[b])]
            i = int(np.argmin((tr[:, 4] - st[b, 0]) ** 2 + (tr[:, 5] - st[b, 1]) ** 2))
            sq = tr[i, 6] + s_fit
            dx = np.interp(sq, tr[:, 6], tr[:, 4]) - st[b, 0]; dy = np.interp(sq, tr[:, 6], tr[:, 5]) - st[b, 1]
            c, s_ = np.cos(st[b, 2]), np.sin(st[b, 2])
            xw[b] = c * dx + s_ * dy; yw[b] = -s_ * dx + c * dy
        K, psi_start = frenet_ref.fit_windows(xw, yw, window)
        kpoly[:] = K
        state[:, 0] = 0.0
        state[:, 1] = -(-np.sin(psi_start) * xw[:, 0] + np.cos(psi_start) * yw[:, 0]) if ey_from_path else 0.0
        state[:, 2] = -psi_start
        state[:, 3] = st[:, 3]
        out = solver.solve_batch(state, kpoly, u_curr, v_des=np.full(B, float(target_vel)), warm=warm)
        sim.mpc_cmd(out["u0"][:, 0], out["u0"][:, 1])
        u_curr[:, 0] = out["u0"][:, 1]; u_curr[:, 1] = out["u0"][:, 0]
        log[t, :, 0:4] = st
        log[t, :, 4] = out["u0"][:, 0]; log[t, :, 5] = out["u0"][:, 1]
        log[t, :, 6] = out["status"]; log[t, :, 7] = out["iters"]
    if own:
        solver.close()
    return {"log": log, "final_state": sim.full_state()}
