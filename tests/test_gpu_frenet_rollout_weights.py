"""GPU tests of per-vehicle cost weights in the Frenet closed loop (mpcb200_rollout_frenet_w) through the C ABI.

Which instantiation each case reaches (csrc/mpc_b200.cu: rollout_enqueue):
  fused      mpc_rollout_frenet_kernel<0, 1> (<1, 1> with metrics): rollout_group_frenet stages the vehicle's row in shared memory
  pipeline   rollout_frenet_ref_kernel + rollout_solve_tpp_kernel<1, 1>, set_large_batch_path(1): the slot reads its vehicle's row

1. Iterate for iterate against oracle.closed_loop_frenet with each vehicle's own row, in the scheme of test_gpu_frenet_closed_loop.py:
   max_iter = 3 (equal statuses and iteration counts, poses and commands within the row's bar relative to max(1, |x|)), then the
   default cap (equal statuses, iterations within one, commands within U_BAR).
2. Rows equal to the handle's weights reproduce rollout_frenet; 3. a fleet of mixed rows equals the same rows run as separate
   set_cost_frenet + rollout_frenet fleets.  Both in both forms, with equal statuses and iterations and log / final state within
   SAME_BAR (the bar of the XY test_weighted_rollout_matches_oracle_closed_loop).
4. With metrics: the log of the same call without metrics bit for bit, and closed_loop.tracking_metrics of it; 5. launch counts.
6. Argument errors (MPCB200_EINVAL naming the entry point), after which the handle still serves a valid call.
7. Two GPUs: the fleet runs on devices[0] and gives the one-GPU result bit for bit.
`pytest -s` prints the observed table."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

T = 6
U_BAR = 1e-8       # uncapped: |du|
SAME_BAR = 1e-12   # equal rows / mixed rows against the unweighted loop: |d log|, |d final|; observed on a B200 (1,000 W): 0 except
#                    mixed_rows_pipeline 4.4e-16.  At 16,384 vehicles x 200 periods the pipeline's logs part (DESIGN.md section 3.4)
W_DEFAULT = np.array([9.0, 10.0, 0.5, 100.0, 1000.0, 0.0, 0.0])   # MKZMPCPathFollowerFrenet.jl:51-58, set_cost_frenet's order
EXACT = [0, 3, 5, 8, 9, 10, 11]

# id: (N, fleet size (7: over the three paths), per-period pipeline)
ROWS = {
    "fused_N3":     (3, 3, False),
    "fused_N8":     (8, 3, False),
    "fused_N20":    (20, 3, False),
    "fused_N31":    (31, 3, False),
    "pipeline_N8":  (8, 3, True),
    "pipeline_N31": (31, 3, True),
    "fleet7":       (8, 7, False),
}

# row id -> bar: 10x the largest relative difference observed on a B200 (1,000 W power limit), rounded up to one digit
BARS = {
    "fleet7":       7e-14,    # observed 6.19e-15
    "fused_N20":    7e-15,    # observed 6.87e-16
    "fused_N3":     1e-14,    # observed 9.99e-16
    "fused_N31":    9e-13,    # observed 8.96e-14
    "fused_N8":     2e-14,    # observed 1.69e-15
    "pipeline_N31": 8e-13,    # observed 7.51e-14
    "pipeline_N8":  9e-15,    # observed 8.22e-16
}

OBSERVED = {}


def observe(row, d, bar):
    OBSERVED[row] = (max(OBSERVED.get(row, (0.0,))[0], float(d)) if d == d else float("nan"), bar)
    assert d <= bar, (row, d, bar)


@pytest.fixture(scope="module", autouse=True)
def _print_observed():
    yield
    for row in sorted(OBSERVED):
        print("observed %-22s %.2e  (bar %.0e)" % (row, OBSERVED[row][0], OBSERVED[row][1]))


@pytest.fixture(scope="module")
def capi():
    from mkz_mpc_path_follower_b200 import capi as c
    c.lib()
    return c


@pytest.fixture(scope="module")
def tables():
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    return [GPSRefTrajectory(mat_filename=p).trajectory for p in (1, 2, 3)]


def weight_rows(B, seed):
    from test_frenet_weights_emu import weight_rows as rows
    return rows(B, seed)


def solver(capi, tables, N=8, pipeline=False, max_iter=None, devices=None):
    kw = {} if max_iter is None else {"max_iter": max_iter}
    s = capi.FrenetSolver(N, devices=devices, **kw)
    s.set_large_batch_path(1 if pipeline else 0)
    for i, tr in enumerate(tables):
        s.set_path(i, tr)
    return s


def fleet(tables, per_path=6, seed=1):
    """per_path vehicles near random samples of each path (with 40 m of path ahead), beside it and turned a little; ids 0..2."""
    rng = np.random.default_rng(seed)
    poses, pid = [], []
    for p, tr in enumerate(tables):
        for i in rng.integers(0, tr.shape[0] - 2000, size=per_path):
            poses.append(tr[i, [4, 5, 3]] + rng.normal(scale=[0.3, 0.3, 0.03]))
            pid.append(p)
    return np.array(poses), np.array(pid, dtype=np.int32)


def same_loop(name, a, b):
    """Equal statuses and iterations, log and final state within SAME_BAR."""
    assert np.array_equal(a["log"][:, :, 6:8], b["log"][:, :, 6:8]), name
    d = max(np.abs(a["log"] - b["log"]).max(), np.abs(a["final_state"] - b["final_state"]).max())
    observe(name, d, SAME_BAR)


@pytest.mark.parametrize("row", list(ROWS))
def test_weighted_rollout_iterates(capi, oracle, tables, row):
    from test_frenet_closed_loop_emu import loop_fleet
    N, B, pipeline = ROWS[row]
    pose0, path_of = loop_fleet(tables, B, seed=N)
    rows = weight_rows(B, seed=N)
    for max_iter in (3, None):
        s = solver(capi, tables, N, pipeline, max_iter)
        cap = s.cfg.max_iter
        glog = s.rollout(pose0, path_of, T, weights=rows)["log"]
        assert s.stats()["kernel_launches"] == (3 * T + 1 if pipeline else 1)
        s.close()
        olog = np.stack([oracle.closed_loop_frenet(oracle.default_cfg_frenet(N, weights=(0.0,) + tuple(rows[v]), max_iter=cap),
                                                   tables[path_of[v]], pose0[v], T, 40.0, 8.0, True) for v in range(B)], axis=1)
        assert np.array_equal(glog[:, :, 6], olog[:, :, 6]), (row, glog[:, :, 6], olog[:, :, 6])
        if max_iter is not None:
            assert np.array_equal(glog[:, :, 7], olog[:, :, 7]), (row, glog[:, :, 7], olog[:, :, 7])
            assert (olog[:, :, 6] == 3).mean() >= 0.9, row
            observe(row, (np.abs(glog[:, :, 0:6] - olog[:, :, 0:6]) / np.maximum(1.0, np.abs(olog[:, :, 0:6]))).max(), BARS[row])
        else:
            assert (olog[:, :, 6] == 0).mean() >= 0.9, row
            assert np.abs(glog[:, :, 7] - olog[:, :, 7]).max() <= 1, (row, glog[:, :, 7], olog[:, :, 7])
            observe(row + "_du", np.abs(glog[:, :, 4:6] - olog[:, :, 4:6]).max(), U_BAR)


@pytest.mark.parametrize("pipeline", [False, True], ids=["fused", "pipeline"])
def test_equal_rows_reproduce_rollout_frenet(capi, tables, pipeline):
    s = solver(capi, tables, pipeline=pipeline)
    poses, pid = fleet(tables)
    T_ = 60
    plain = s.rollout(poses, pid, T_)
    eq = s.rollout(poses, pid, T_, weights=np.tile(W_DEFAULT, (len(poses), 1)))
    same_loop("equal_rows_" + ("pipeline" if pipeline else "fused"), eq, plain)
    s.close()


@pytest.mark.parametrize("pipeline", [False, True], ids=["fused", "pipeline"])
def test_mixed_rows_equal_separate_fleets(capi, tables, pipeline):
    poses, pid = fleet(tables, per_path=8, seed=2)
    rows4 = weight_rows(4, seed=3)
    which = np.arange(len(poses)) % 4
    T_ = 40
    s = solver(capi, tables, pipeline=pipeline)
    mixed = s.rollout(poses, pid, T_, weights=rows4[which])
    for r in range(4):
        sel = which == r
        s.set_cost(rows4[r])
        sep = s.rollout(poses[sel], pid[sel], T_)
        part = {"log": mixed["log"][:, sel], "final_state": mixed["final_state"][sel]}
        same_loop("mixed_rows_" + ("pipeline" if pipeline else "fused"), part, sep)
    s.close()


@pytest.mark.parametrize("pipeline", [False, True], ids=["fused", "pipeline"])
def test_metrics_with_rows(capi, tables, pipeline):
    from mkz_mpc_path_follower_b200.closed_loop import tracking_metrics
    s = solver(capi, tables, pipeline=pipeline)
    poses, pid = fleet(tables, seed=4)
    rows = weight_rows(len(poses), seed=5)
    T_ = 30
    plain = s.rollout(poses, pid, T_, weights=rows)
    assert s.stats()["kernel_launches"] == (3 * T_ + 1 if pipeline else 1)
    out = s.rollout(poses, pid, T_, weights=rows, metrics=True)
    assert s.stats()["kernel_launches"] == (4 * T_ + 2 if pipeline else 2)
    assert np.array_equal(out["log"], plain["log"]) and np.array_equal(out["final_state"], plain["final_state"])
    ref = np.empty((len(poses), 12))
    for p, tr in enumerate(tables):
        ref[pid == p] = tracking_metrics(out["log"][:, pid == p, :], tr)
    met = out["metrics"]
    assert np.array_equal(met[:, EXACT], ref[:, EXACT], equal_nan=True)
    rest = [f for f in range(12) if f not in EXACT]
    assert (np.abs(met[:, rest] - ref[:, rest]) <= 1e-12 * np.maximum(np.abs(ref[:, rest]), 1e-300)).all()
    assert (met[:, 0] == T_).all() and (met[:, 11] == -1).all()
    nolog = s.rollout(poses, pid, T_, weights=rows, metrics=True, want_log=False)
    assert nolog["log"] is None and np.array_equal(nolog["metrics"], met, equal_nan=True)
    s.close()


def test_argument_errors(capi, tables):
    """Each refused call returns MPCB200_EINVAL with mpcb200_rollout_frenet_w in the message; the handle then still serves."""
    L = capi.lib()
    dp = C.POINTER(C.c_double)
    poses, pid = fleet(tables)
    B = len(poses)
    pp, ip = poses.ctypes.data_as(dp), pid.ctypes.data_as(C.POINTER(C.c_int32))
    rows = weight_rows(B, seed=7)
    s = solver(capi, tables)
    good = s.rollout(poses, pid, 5, weights=rows)

    def refused(h, w, window=40.0, what=""):
        log = np.full((5, B, 8), 7.0)
        rc = L.mpcb200_rollout_frenet_w(h, B, 5, pp, ip, window, 8.0, 1, None if w is None else w.ctypes.data_as(dp),
                                        log.ctypes.data_as(dp), None, None)
        msg = L.mpcb200_last_error(h).decode()
        assert rc == -1 and "mpcb200_rollout_frenet_w" in msg and what in msg, (rc, msg)

    for v in (float("nan"), -0.5):
        bad = rows.copy()
        bad[2, 3] = v
        refused(s._h, bad, what="weight 3 of vehicle 2")
        assert np.array_equal(s.rollout(poses, pid, 5, weights=rows)["log"], good["log"])
    refused(s._h, None, what="w is required")
    refused(s._h, rows, window=3.0, what="window")
    refused(s._h, rows, window=501.0, what="window")
    assert np.array_equal(s.rollout(poses, pid, 5, weights=rows)["log"], good["log"])
    xy = capi.Solver(8)
    xy.set_path(0, tables[0])
    refused(xy._h, rows, what="mpcb200_create_frenet")
    xy.close()
    long = solver(capi, tables, N=40)
    refused(long._h, rows, what="N <= 31")
    long.close()
    with pytest.raises(ValueError):
        s.rollout(poses, pid, 5, weights=rows[:, :6])
    with pytest.raises(ValueError):
        s.rollout(poses, pid, 5, weights=rows[1:])
    assert np.array_equal(s.rollout(poses, pid, 5, weights=rows)["log"], good["log"])
    s.close()


def test_two_devices_as_one(capi, tables):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    poses, pid = fleet(tables, per_path=20, seed=9)
    rows = weight_rows(len(poses), seed=9)
    out = {}
    for name, devices in (("one", [0]), ("multi", [0, 1])):
        s = solver(capi, tables, devices=devices)
        out[name] = s.rollout(poses, pid, 30, weights=rows, metrics=True)
        out[name + "_launches"] = s.stats()["kernel_launches"]
        s.close()
    assert out["one_launches"] == out["multi_launches"] == 2   # the fused kernel and the metrics rows, on one device
    for k in ("log", "final_state", "metrics"):
        assert np.array_equal(out["one"][k], out["multi"][k], equal_nan=True), k
