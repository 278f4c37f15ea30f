"""GPU tests of per-problem cost weights (mpcb200_solve_batch_w, mpcb200_solve_batch_frenet_w, mpcb200_rollout_w) through the C
ABI: oracle parity with each problem's own weights in both device layouts, agreement with the unweighted entry points, device
pointers, the small-batch graph cache, multi-GPU slicing, bad rows and closed-loop rollouts.  Tolerances as in
tests/test_gpu_parity.py (BASELINE.json): same status, |du| <= 1e-5, relative cost <= 1e-6."""
import numpy as np
import pytest

from mkz_mpc_path_follower_b200 import workload as W

pytestmark = pytest.mark.gpu

U_TOL = 1e-5
COST_RTOL = 1e-6
W_XY = np.array([9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0])
W_FRENET = np.array([9.0, 10.0, 0.5, 100.0, 1000.0, 0.0, 0.0])


@pytest.fixture(scope="module")
def capi():
    from mkz_mpc_path_follower_b200 import capi as c
    c.lib()
    return c


def weight_rows(B, n, seed):
    """Log-uniform in [0.1x, 10x] the module defaults (around 1 where the default is 0), row 0 the defaults, row 1 ca = cd = 0."""
    rng = np.random.default_rng(seed)
    base = (W_XY if n == 8 else W_FRENET).copy()
    rows = np.where(base > 0, base, 1.0) * 10.0 ** rng.uniform(-1.0, 1.0, size=(B, n))
    rows[0] = base
    rows[1, -2:] = 0.0
    return rows


def oracle_rows(oracle, solver, rows, frenet, *inputs):
    c = solver.cfg
    outs = []
    for b in range(rows.shape[0]):
        if frenet:
            cfg = oracle.default_cfg_frenet(c.N, weights=np.concatenate([[0.0], rows[b]]), tol=c.tol, max_iter=c.max_iter)
            outs.append(oracle.solve_batch_frenet(cfg, *[a[b:b + 1] for a in inputs]))
        else:
            cfg = oracle.default_cfg(c.N, weights=rows[b], tol=c.tol, max_iter=c.max_iter)
            outs.append(oracle.solve_batch(cfg, *[a[b:b + 1] for a in inputs]))
    return {k: np.concatenate([o[k] for o in outs]) for k in ("u0", "status", "iters", "cost")}


def compare(g, o, min_conv=0.8, max_status_mismatch=0):
    """Statuses may differ only for long solves: the rounding of the Riccati recursion against the oracle's dense LDL' shows
    after ~100 iterations, where a solve near the 200-iteration cap can end on the other side of it."""
    mism = np.nonzero(g["status"] != o["status"])[0]
    assert mism.size <= max_status_mismatch + 2 and (o["iters"][mism] >= 100).all(), (mism, o["iters"][mism], g["iters"][mism])
    ok = (o["status"] == 0) & (g["status"] == 0)
    assert ok.mean() >= min_conv
    assert np.abs(g["u0"] - o["u0"])[ok].max() <= U_TOL
    assert (np.abs(g["cost"] - o["cost"])[ok] / np.maximum(1.0, np.abs(o["cost"][ok]))).max() <= COST_RTOL


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("N,B", [(8, 256), (20, 192), (40, 24)])
def test_weighted_xy_matches_oracle(capi, oracle, layout, N, B):
    s = capi.Solver(N)
    s.set_large_batch_path(layout)
    b = W.make_batch(B, N)
    rows = weight_rows(B, 8, seed=N)
    g = s.solve_batch(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"], weights=rows)
    o = oracle_rows(oracle, s, rows, False, b["state"], b["ref"], b["v_des"], b["u_prev"])
    compare(g, o, min_conv=0.8 if N <= 20 else 0.5, max_status_mismatch=0 if N <= 20 else 1)


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("N,B", [(8, 128), (20, 96)])
def test_weighted_frenet_matches_oracle(capi, oracle, layout, N, B):
    s = capi.FrenetSolver(N)
    s.set_large_batch_path(layout)
    b = W.make_frenet_batch(B, N)
    rows = weight_rows(B, 7, seed=100 + N)
    g = s.solve_batch(b["state"], b["kpoly"], b["u_prev"], v_des=b["v_des"], weights=rows)
    o = oracle_rows(oracle, s, rows, True, b["state"], b["kpoly"], b["v_des"], b["u_prev"])
    compare(g, o)


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("B", [16, 300])
def test_equal_rows_match_unweighted(capi, layout, B):
    """Every row equal to the handle's weights: the same solve as solve_batch.  The PW = 1 kernels read the weights from shared
    memory / the row instead of the kernel parameter and compute the same expressions in the same order: bit-identical."""
    N = 8
    s = capi.Solver(N)
    s.set_large_batch_path(layout)
    b = W.make_batch(B, N)
    u = s.solve_batch(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"], want_traj=True)
    ru = s.restorations(B)
    g = s.solve_batch(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"], want_traj=True, weights=np.tile(W_XY, (B, 1)))
    assert (g["status"] == u["status"]).all() and (g["iters"] == u["iters"]).all()
    assert (s.restorations(B) == ru).all()
    for k in ("u0", "cost", "traj"):
        assert np.abs(g[k] - u[k]).max() <= 1e-12, k


@pytest.mark.parametrize("layout", [0, 1])
def test_mixed_batch_equals_set_cost_runs(capi, layout):
    N, B = 8, 256
    b = W.make_batch(B, N)
    vecs = weight_rows(4, 8, seed=3)
    which = np.arange(B) % 4
    s = capi.Solver(N)
    s.set_large_batch_path(layout)
    g = s.solve_batch(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"], weights=vecs[which])
    for j in range(4):
        m = which == j
        r = capi.Solver(N)
        r.set_large_batch_path(layout)
        r.set_cost(vecs[j])
        u = r.solve_batch(b["state"][m], b["ref"][m], b["u_prev"][m], v_des=b["v_des"][m])
        assert (u["status"] == g["status"][m]).all() and (u["iters"] == g["iters"][m]).all()
        assert np.abs(u["u0"] - g["u0"][m]).max() <= 1e-12


@pytest.mark.parametrize("frenet", [False, True])
def test_device_pointers_and_bad_rows(capi, frenet):
    """Torch tensors give what host arrays give; a negative or NaN row on the device gives that problem MPCB200_ERROR and zero
    commands, its neighbours are unaffected; the same rows from the host are refused."""
    import torch
    N, B = 8, 96
    if frenet:
        s, b, n = capi.FrenetSolver(N), W.make_frenet_batch(B, N), 7
        ref = b["kpoly"]
    else:
        s, b, n = capi.Solver(N), W.make_batch(B, N), 8
        ref = b["ref"]
    rows = weight_rows(B, n, seed=9)
    h = s.solve_batch(b["state"], ref, b["u_prev"], v_des=b["v_des"], weights=rows)
    bad = rows.copy()
    bad[5, 2] = -1.0
    bad[17, 0] = np.nan
    with pytest.raises(capi.MpcB200Error) as ei:
        s.solve_batch(b["state"], ref, b["u_prev"], v_des=b["v_des"], weights=bad)
    assert ei.value.code == -1 and "problem 5" in str(ei.value)
    dev = torch.device("cuda:0")
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev)
    for rw, badset in ((rows, []), (bad, [5, 17])):
        u0 = torch.zeros((B, 2), dtype=torch.float64, device=dev); cost = torch.zeros(B, dtype=torch.float64, device=dev)
        status = torch.zeros(B, dtype=torch.int32, device=dev); iters = torch.zeros(B, dtype=torch.int32, device=dev)
        s.solve_batch_device(B, t(b["state"]), t(ref), t(b["u_prev"]), u0, v_des=t(b["v_des"]), cost=cost, status=status, iters=iters,
                             weights=t(rw))
        torch.cuda.synchronize()
        g = {"u0": u0.cpu().numpy(), "cost": cost.cpu().numpy(), "status": status.cpu().numpy(), "iters": iters.cpu().numpy()}
        good = ~np.isin(np.arange(B), badset)
        assert (g["status"][good] == h["status"][good]).all() and (g["iters"][good] == h["iters"][good]).all()
        assert np.abs(g["u0"][good] - h["u0"][good]).max() <= 1e-12
        if badset:
            assert (g["status"][~good] == capi.ERROR).all() and (g["u0"][~good] == 0).all()
            assert (g["iters"][~good] == 0).all() and (g["cost"][~good] == 0).all()
    with pytest.raises(ValueError):
        s.solve_batch(b["state"], ref, b["u_prev"], weights=rows[:, :n - 1])


def test_small_batch_graph_cache(capi):
    """B = 16 (the packed small-batch path, captured as a CUDA graph per shape): unweighted, weighted with other rows, unweighted
    again -- each equal to a fresh handle's answer."""
    N, B = 8, 16
    b = W.make_batch(B, N)
    rows = weight_rows(B, 8, seed=21)
    rows2 = weight_rows(B, 8, seed=22)
    s = capi.Solver(N)
    args = (b["state"], b["ref"], b["u_prev"])
    seq = [None, rows, rows2, None]
    got = [s.solve_batch(*args, v_des=b["v_des"], weights=w) for w in seq]
    for w, g in zip(seq, got):
        f = capi.Solver(N).solve_batch(*args, v_des=b["v_des"], weights=w)
        assert (g["status"] == f["status"]).all() and np.array_equal(g["u0"], f["u0"]) and np.array_equal(g["cost"], f["cost"])
    assert not np.array_equal(got[1]["u0"], got[2]["u0"])


def test_multi_gpu_slices_the_rows(capi):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    N, B = 8, 1000
    b = W.make_batch(B, N)
    rows = weight_rows(B, 8, seed=31)
    one = capi.Solver(N).solve_batch(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"], weights=rows)
    two = capi.Solver(N, devices=[0, 1]).solve_batch(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"], weights=rows)
    for k in ("u0", "cost", "status", "iters"):
        assert np.array_equal(one[k], two[k]), k


@pytest.mark.parametrize("pipeline", [False, True])
def test_weighted_rollout_matches_oracle_closed_loop(capi, oracle, pipeline):
    """rollout_w against the oracle's closed loop with each vehicle's own weights, for the fused kernel and the per-period pipeline
    (set_large_batch_path(1)); rows all equal to the handle's weights reproduce rollout."""
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    s = capi.Solver(8)
    if pipeline:
        s.set_large_batch_path(1)
    trajs = [GPSRefTrajectory(mat_filename=p) for p in (1, 2, 3)]
    for i, g in enumerate(trajs):
        s.set_path(i, g.trajectory)
    rng = np.random.default_rng(4)
    poses, path_of = [(0.0, 3.0, -1.5)], [2]
    for i, g in enumerate(trajs):
        for j in (0, 1500, 4000):
            poses.append((g.trajectory[j, 4] + rng.normal(scale=0.4), g.trajectory[j, 5] + rng.normal(scale=0.4),
                          g.trajectory[j, 3] + rng.normal(scale=0.05)))
            path_of.append(i)
    poses, path_of = np.array(poses), np.array(path_of)
    T = 60
    rows = weight_rows(len(poses), 8, seed=41)
    out = s.rollout(poses, path_of, T, weights=rows)
    for b in range(len(poses)):
        path, keep = oracle.make_path(trajs[path_of[b]].trajectory)
        olog = oracle.closed_loop(oracle.default_cfg(8, weights=rows[b]), path, poses[b], T)
        glog = out["log"][:, b, :]
        assert np.array_equal(glog[:, 6], olog[:, 6]), b
        assert np.abs(glog[:, 4:6] - olog[:, 4:6]).max() <= 1e-5, b
        assert np.abs(glog[:, 0:4] - olog[:, 0:4]).max() <= 1e-4, b
    u = s.rollout(poses, path_of, T)
    e = s.rollout(poses, path_of, T, weights=np.tile(W_XY, (len(poses), 1)))
    assert np.array_equal(u["log"][:, :, 6:8], e["log"][:, :, 6:8]) and np.abs(u["log"] - e["log"]).max() <= 1e-12
    bad = rows.copy()
    bad[2, 7] = -0.5
    with pytest.raises(capi.MpcB200Error):
        s.rollout(poses, path_of, T, weights=bad)
