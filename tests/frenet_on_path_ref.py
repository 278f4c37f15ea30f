"""TEST ONLY: the Frenet node's reference step for one pose with nothing from the library -- the per-period reference of
oracle.closed_loop_frenet on its own (gazebo_sim_mpc_cmd_pub_frenet.jl:112-130 with nav_msgs_path_frenet.py:44-86): the nearest
sample by np.argmin, the next `window` metres every 0.5 m by np.interp seen from the vehicle, oracle.frenet_fit, and e_y.
test_frenet_on_path_emu.py checks that a loop built on it reproduces oracle.closed_loop_frenet bit for bit."""
import math

import numpy as np


def frenet_on_path(O, traj_table, pose, window, ey_from_path=True):
    """O: the oracle module; traj_table: the (n,7) table of GPSRefTrajectory.trajectory; pose (X, Y, psi, v).  Returns
    (K (4,) highest degree first, state (4,) = (0, e_y, -psi_start, v)), as closed_loop_frenet gives them to solve_batch_frenet."""
    Xp, Yp, sp = (np.ascontiguousarray(traj_table[:, i], dtype=np.float64) for i in (4, 5, 6))
    X, Y, psi, v = (float(x) for x in pose)
    i = int(np.argmin((Xp - X) ** 2 + (Yp - Y) ** 2))
    sq = sp[i] + np.arange(0.0, window, 0.5)
    dx = np.interp(sq, sp, Xp) - X; dy = np.interp(sq, sp, Yp) - Y
    c, s = np.cos(psi), np.sin(psi)
    xw = c * dx + s * dy; yw = -s * dx + c * dy
    K, psi_start = O.frenet_fit(xw, yw, window)
    ey = -(-np.sin(psi_start) * xw[0] + np.cos(psi_start) * yw[0]) if ey_from_path else 0.0
    return K, np.array([0.0, ey, -psi_start, v])


def frenet_on_path_batch(O, tables, pose, path_of, window, ey_from_path=True):
    """frenet_on_path for B poses (B,4) on tables[path_of[b]]: K (B,4), state (B,4)."""
    r = [frenet_on_path(O, tables[p], q, window, ey_from_path) for q, p in zip(pose, path_of)]
    return np.array([k for k, _ in r]), np.array([s for _, s in r])


def pose_classes(tr, window, v=6.0):
    """(X, Y, psi, v) on the path; 0.7 m and 3 m beside it with heading errors up to +-0.5 rad; across it (heading +-pi/2);
    near the end, so that the window straddles the last sample; 2 km beside the path."""
    j = tr.shape[0] // 2
    nrm = np.array([-np.sin(tr[j, 3]), np.cos(tr[j, 3])])
    poses = [(tr[0, 4], tr[0, 5], tr[0, 3])]
    for off, dpsi in ((0.7, 0.5), (-0.7, -0.3), (3.0, 0.2), (-3.0, -0.5), (0.2, 0.5 * math.pi), (-0.4, -0.5 * math.pi)):
        xy = tr[j, 4:6] + off * nrm
        poses.append((xy[0], xy[1], tr[j, 3] + dpsi))
    je = int(np.searchsorted(tr[:, 6], tr[-1, 6] - 0.5 * min(window, 40.0)))
    poses.append(tuple(tr[je, [4, 5, 3]] + np.array([0.3, -0.2, 0.1])))
    xy = tr[j, 4:6] + 2000.0 * nrm
    poses.append((xy[0], xy[1], tr[j, 3] + 0.1))
    return np.array([(X, Y, p, v + 0.5 * m) for m, (X, Y, p) in enumerate(poses)])


def far_poses(tables, pose, path_of):
    """The poses more than 1 km from their path."""
    return np.array([np.hypot(tables[p][:, 4] - q[0], tables[p][:, 5] - q[1]).min() > 1000.0 for q, p in zip(pose, path_of)])


def batch3(tables, window):
    """The pose classes on all three tables in one batch."""
    pose = np.concatenate([pose_classes(tr, window) for tr in tables])
    path_of = np.repeat(np.arange(3, dtype=np.int32), pose.shape[0] // 3)
    return pose, path_of
