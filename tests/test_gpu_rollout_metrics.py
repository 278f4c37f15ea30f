"""GPU tests of the rollout tracking metrics (mpcb200_rollout_metrics, mpcb200_rollout_frenet_metrics) through the C ABI: every
path that accumulates them -- fused XY at N = 8, 40 and 80 with and without per-vehicle weights, the per-period pipeline, fused and
pipelined Frenet -- against closed_loop.tracking_metrics of the same call's log; log and final state bit-identical to the plain
entry points'; metrics without a log bit-identical to metrics with one; two devices as one; the argument errors."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EXACT = [0, 3, 5, 8, 9, 10, 11]
W_XY = np.array([9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0])


@pytest.fixture(scope="module")
def capi():
    from mkz_mpc_path_follower_b200 import capi as c
    c.lib()
    return c


@pytest.fixture(scope="module")
def trajs():
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    return [GPSRefTrajectory(mat_filename=p) for p in (1, 2, 3)]


def fleet(trajs, N=8, per_path=6, seed=1):
    """On each path: one vehicle on the last sample (stop in period 0), one a little more than the horizon before the end, one
    across the -pi / +pi jump of the recorded heading, the rest near random samples; path ids 0..2."""
    rng = np.random.default_rng(seed)
    poses, pid = [], []
    for p, g in enumerate(trajs):
        tr = g.trajectory
        n = tr.shape[0]
        j = int(np.nonzero(np.abs(np.diff(tr[:, 3])) > 3.0)[0][0])
        idx = [n - 1, n - 1 - 20 * N - 5, j] + [int(x) for x in rng.integers(0, n - 2000, size=per_path - 3)]
        for i in idx:
            poses.append(tr[i, [4, 5, 3]] + (0.0 if i >= n - 1 - 20 * N - 5 else rng.normal(scale=[0.3, 0.3, 0.03])))
            pid.append(p)
    return np.array(poses), np.array(pid, dtype=np.int32)


def solver(capi, trajs, frenet=False, N=8, pipeline=False, devices=None):
    s = capi.FrenetSolver(N, devices=devices) if frenet else capi.Solver(N, devices=devices)
    s.set_large_batch_path(1 if pipeline else 0)
    for i, g in enumerate(trajs):
        s.set_path(i, g.trajectory)
    return s


def host_metrics(log, pid, trajs):
    from mkz_mpc_path_follower_b200.closed_loop import tracking_metrics
    out = np.empty((log.shape[1], 12))
    for p, g in enumerate(trajs):
        m = pid == p
        out[m] = tracking_metrics(log[:, m, :], g.trajectory)
    return out


def check(met, ref):
    assert np.array_equal(met[:, EXACT], ref[:, EXACT], equal_nan=True)
    rest = [f for f in range(12) if f not in EXACT]
    assert (np.abs(met[:, rest] - ref[:, rest]) <= 1e-12 * np.maximum(np.abs(ref[:, rest]), 1e-300)).all()


@pytest.mark.parametrize("N,pw,pipeline", [(8, False, False), (8, True, False), (40, False, False), (40, True, False), (80, False, False),
                                           (8, False, True), (8, True, True)])
def test_xy_metrics(capi, trajs, N, pw, pipeline):
    s = solver(capi, trajs, N=N, pipeline=pipeline)
    poses, pid = fleet(trajs, N)
    T = 40 if N == 8 else 15
    w = W_XY * 10.0 ** np.random.default_rng(N).uniform(-0.5, 0.5, size=(len(poses), 8)) if pw else None
    plain = s.rollout(poses, pid, T, weights=w)
    out = s.rollout(poses, pid, T, weights=w, metrics=True)
    launches = s.stats()["kernel_launches"]
    assert launches == (4 * T + 2 if pipeline else 2)
    assert np.array_equal(out["log"], plain["log"]) and np.array_equal(out["final_state"], plain["final_state"])
    check(out["metrics"], host_metrics(out["log"], pid, trajs))
    nolog = s.rollout(poses, pid, T, weights=w, metrics=True, want_log=False)
    assert nolog["log"] is None
    assert np.array_equal(nolog["metrics"], out["metrics"], equal_nan=True) and np.array_equal(nolog["final_state"], out["final_state"])
    m = out["metrics"]
    last = (np.arange(len(poses)) % 6 == 0) & (pid == 0)
    assert (m[last, 0] == 0).all() and (m[last, 11] == 0).all() and np.isnan(m[last, 10]).all()
    if N == 8:   # (path 1; at longer horizons the vehicles do not reach the end of the horizon within T)
        mid = (np.arange(len(poses)) % 6 == 1) & (pid == 0)
        assert ((m[mid, 11] > 0) & (m[mid, 11] < T) & (m[mid, 0] == m[mid, 11])).all()
    assert (m[np.arange(len(poses)) % 6 == 2, 5] < 0.5).all()   # heading error wrapped across the recorded -pi / +pi jump


@pytest.mark.parametrize("pipeline", [False, True])
def test_frenet_metrics(capi, trajs, pipeline):
    s = solver(capi, trajs, frenet=True, pipeline=pipeline)
    poses, pid = fleet(trajs)
    keep = np.arange(len(poses)) % 6 >= 2   # vehicles with 40 m of path ahead
    poses, pid = poses[keep], pid[keep]
    T = 30
    plain = s.rollout(poses, pid, T)
    out = s.rollout(poses, pid, T, metrics=True)
    assert s.stats()["kernel_launches"] == (4 * T + 2 if pipeline else 2)
    assert np.array_equal(out["log"], plain["log"]) and np.array_equal(out["final_state"], plain["final_state"])
    check(out["metrics"], host_metrics(out["log"], pid, trajs))
    assert (out["metrics"][:, 0] == T).all() and (out["metrics"][:, 11] == -1).all()
    nolog = s.rollout(poses, pid, T, metrics=True, want_log=False)
    assert np.array_equal(nolog["metrics"], out["metrics"], equal_nan=True)


def test_two_devices_as_one(capi, trajs):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    poses, pid = fleet(trajs, per_path=40)
    one = solver(capi, trajs).rollout(poses, pid, 30, metrics=True)
    two = solver(capi, trajs, devices=[0, 1]).rollout(poses, pid, 30, metrics=True)
    for k in ("log", "final_state", "metrics"):
        assert np.array_equal(one[k], two[k], equal_nan=True), k


def test_argument_errors(capi, trajs):
    """A NULL metrics buffer; the XY entry point (the one with w) on a Frenet handle; nothing written with T = 0."""
    L = capi.lib()
    dp = C.POINTER(C.c_double)
    poses, pid = fleet(trajs)
    B = len(poses)
    pp, ip = poses.ctypes.data_as(dp), pid.ctypes.data_as(C.POINTER(C.c_int32))
    w = np.tile(W_XY, (B, 1))
    met = np.full((B, 12), 7.0)
    s = solver(capi, trajs)
    assert L.mpcb200_rollout_metrics(s._h, B, 5, pp, ip, 1, 1.0, None, None, None, None) == -1
    f = solver(capi, trajs, frenet=True)
    assert L.mpcb200_rollout_frenet_metrics(f._h, B, 5, pp, ip, 40.0, 8.0, 1, None, None, None) == -1
    assert L.mpcb200_rollout_metrics(f._h, B, 5, pp, ip, 1, 1.0, w.ctypes.data_as(dp), None, None, met.ctypes.data_as(dp)) == -1
    assert L.mpcb200_rollout_metrics(s._h, B, 0, pp, ip, 1, 1.0, None, None, None, met.ctypes.data_as(dp)) == 0
    assert (met == 7.0).all()
    with pytest.raises(capi.MpcB200Error):
        f.rollout(poses, pid, 5, metrics=True, window=1.0)
