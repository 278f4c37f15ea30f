"""CPU check of the rollout tracking metrics (mpcb200_rollout_metrics, mpcb200_rollout_frenet_metrics): the MET = 1 instantiations of
the kernel sources on the warp emulator (tests/emu/emu_metrics.py) -- fused XY at one- and two-warp horizons with and without
per-vehicle weights, the per-period pipeline with its metrics kernel, fused Frenet -- against closed_loop.tracking_metrics of the same
run's log, and that log against the loop without metrics.  Then tracking_metrics itself on a hand-built log."""
import os
import sys

import numpy as np
import pytest

from mkz_mpc_path_follower_b200 import capi
from mkz_mpc_path_follower_b200.closed_loop import tracking_metrics
from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

EXACT = [0, 3, 5, 8, 9, 10, 11]   # counts, maxima, s_last, stop_period
W_XY = np.array([9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0])


def check_metrics(met, ref):
    assert met.shape == ref.shape == (ref.shape[0], len(capi.ROLLOUT_METRICS))
    assert np.array_equal(met[:, EXACT], ref[:, EXACT], equal_nan=True), (met[:, EXACT], ref[:, EXACT])
    rest = [f for f in range(12) if f not in EXACT]
    assert (np.abs(met[:, rest] - ref[:, rest]) <= 1e-12 * np.maximum(np.abs(ref[:, rest]), 1e-300)).all(), (met[:, rest], ref[:, rest])


@pytest.fixture(scope="module")
def path1():
    return GPSRefTrajectory(mat_filename=1).trajectory


def xy_fleet(tr, N=8):
    """Vehicle 0 on the last path sample (stop_cmd in period 0), 1 a little more than the horizon (N x 0.2 s, 100 samples a second)
    before the end (latches mid-run), 2 across the -pi / +pi jump of the recorded heading, 3 and 4 off the path with heading errors."""
    n = tr.shape[0]
    j = int(np.nonzero(np.abs(np.diff(tr[:, 3])) > 3.0)[0][0])
    rows = [tr[n - 1, [4, 5, 3]], tr[n - 1 - 20 * N - 5, [4, 5, 3]], tr[j, [4, 5, 3]] + [0.05, -0.05, 0.0],
            tr[900, [4, 5, 3]] + [0.4, -0.3, 0.08], tr[2500, [4, 5, 3]] + [-0.3, 0.2, -0.05]]
    return np.array(rows)


@pytest.mark.parametrize("N,pw", [(8, False), (8, True), (40, False), (40, True)])
def test_fused_xy_metrics_match_log(oracle, path1, N, pw):
    """rollout_group<W, PW, 1> (W = 1 at N = 8, W = 2 at N = 40): log and final state as without metrics, metrics as
    tracking_metrics of that log, and the stop cases of the fleet as the log shows them."""
    import emu as E
    import emu_metrics as EM
    import emu_weights as EW
    cfg = oracle.default_cfg(N)
    k = E.kcfg_from_oracle(cfg)
    seed = oracle.module_load_solution(cfg)
    poses = xy_fleet(path1, N)
    T = 12 if N == 8 else 6
    rng = np.random.default_rng(N)
    w = (W_XY * 10.0 ** rng.uniform(-0.5, 0.5, size=(len(poses), 8))) if pw else None
    log, final, met = EM.rollout_metrics(k, path1, poses, T, w=w, pw=pw, warm0=seed)
    if pw:
        plog, pfinal = EW.rollout_w(k, path1, poses, T, w, warm0=seed)
    else:
        plog, pfinal = E.rollout(k, path1, poses, T, warm0=seed)
    assert np.array_equal(log, plog) and np.array_equal(final, pfinal)
    check_metrics(met, tracking_metrics(log, path1))
    assert met[0, 0] == 0 and np.isnan(met[0, 10]) and met[0, 11] == 0 and (met[0, 1:10] == 0).all()
    if N == 8:   # (at N = 40 the vehicles starting from rest do not reach the end of the 8 s horizon within the test's periods)
        assert 0 < met[1, 0] < T and met[1, 11] == met[1, 0] and (log[int(met[1, 11]):, 1, 6] == -1).all()
    assert (met[2:, 0] == T).all() and (met[2:, 11] == -1).all()
    assert met[2, 5] < 0.5   # wrapped: the recorded heading jumps by 2 pi next to this vehicle


def test_pipeline_metrics_match_log(oracle, path1):
    """The per-period pipeline (plant, waypoints, thread-per-problem solve) with the metrics kernel's source (metrics_period):
    log as without metrics, metrics as tracking_metrics of the log."""
    import emu as E
    import emu_metrics as EM
    cfg = oracle.default_cfg(8)
    k = E.kcfg_from_oracle(cfg)
    seed = oracle.module_load_solution(cfg)
    poses = xy_fleet(path1)
    T = 12
    log, final, met = EM.rollout_metrics(k, path1, poses, T, warm0=seed, tpp=True)
    plog, pfinal = E.rollout(k, path1, poses, T, warm0=seed, tpp=True)
    assert np.array_equal(log, plog) and np.array_equal(final, pfinal)
    check_metrics(met, tracking_metrics(log, path1))
    assert met[0, 0] == 0 and met[0, 11] == 0 and 0 < met[1, 11] < T and (met[2:, 11] == -1).all()


def test_fused_frenet_metrics_match_log(oracle, path1):
    """rollout_group_frenet<1>: every period counts, stop_period -1; log as without metrics."""
    import emu as E
    import emu_metrics as EM
    k = E.kcfg_from_oracle(oracle.default_cfg_frenet(8))
    poses = xy_fleet(path1)[2:]
    T = 8
    log, final, met = EM.rollout_frenet_metrics(k, path1, poses, T)
    plog, pfinal = E.rollout_frenet(k, path1, poses, T)
    assert np.array_equal(log, plog) and np.array_equal(final, pfinal)
    check_metrics(met, tracking_metrics(log, path1))
    assert (met[:, 0] == T).all() and (met[:, 11] == -1).all()


def test_tracking_metrics_hand_built_log():
    """Four samples on the x axis, heading 3.1 (so that a vehicle heading -3.1 is 0.083 rad off, not 6.2), and three vehicles:
    one solving every period, one stopping in period 2, one stopped from period 0."""
    tab = np.zeros((4, 7))
    tab[:, 4] = [0.0, 1.0, 2.0, 3.0]
    tab[:, 3] = 3.1
    tab[:, 6] = [0.0, 1.0, 2.0, 3.0]
    log = np.zeros((3, 3, 8))
    # vehicle 0: (x, y, psi), commands, status, iters per period
    log[:, 0, :] = [[0.1, 0.2, 3.05, 0, 1.0, 0.1, 0, 5], [1.4, -0.1, -3.1, 0, 0.5, 0.0, 3, 7], [2.6, 0.0, 3.1, 0, 0.5, -0.2, 0, 2]]
    log[:, 1, :] = [[2.9, 0.0, 3.1, 0, 2.0, 0.0, 1, 4], [3.0, 0.0, 3.1, 0, 1.0, 0.0, 0, 3], [3.1, 0.0, 3.1, 0, -1.0, 0.0, -1, 0]]
    log[:, 2, :] = [[3.0, 0.5, 3.1, 0, -1.0, 0.0, -1, 0]] * 3
    m = tracking_metrics(log, tab)
    tp = 2.0 * np.pi
    e0 = np.array([np.hypot(0.1, 0.2), np.hypot(0.4, 0.1), np.hypot(0.4, 0.0)])
    h0 = np.array([3.05 - 3.1, (-3.1 - 3.1 + np.pi) % tp - np.pi, 0.0])
    assert m[0, 0] == 3 and np.isclose(m[0, 1], e0.mean()) and np.isclose(m[0, 2], np.sqrt((e0 ** 2).mean()))
    assert np.isclose(m[0, 3], e0.max()) and np.isclose(m[0, 4], np.sqrt((h0 ** 2).mean())) and np.isclose(m[0, 5], np.abs(h0).max())
    assert np.isclose(m[0, 5], tp - 6.2) and np.isclose(m[0, 6], np.sqrt((1.0 + 0.25 + 0.0) / 3)) and np.isclose(m[0, 7], np.sqrt((0.01 + 0.01 + 0.04) / 3))
    assert m[0, 8] == 1 and m[0, 9] == 14 and m[0, 10] == 3.0 and m[0, 11] == -1
    assert m[1, 0] == 2 and np.isclose(m[1, 1], 0.05) and np.isclose(m[1, 3], 0.1) and m[1, 8] == 1 and m[1, 9] == 7
    assert np.isclose(m[1, 6], np.sqrt((4.0 + 1.0) / 2)) and m[1, 10] == 3.0 and m[1, 11] == 2
    assert m[2, 0] == 0 and (m[2, 1:10] == 0).all() and np.isnan(m[2, 10]) and m[2, 11] == 0
