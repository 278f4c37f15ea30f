"""CPU check of per-problem cost weights (mpcb200_solve_batch_w, mpcb200_solve_batch_frenet_w, mpcb200_rollout_w): the PW = 1
instantiations of the kernel sources, run on the warp emulator (tests/emu/emu_weights.py), against the oracle solving each
problem with its own weights, and against unweighted batches with the weights set for the whole batch."""
import os
import sys

import numpy as np
import pytest

from mkz_mpc_path_follower_b200 import workload as W

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

W_XY = np.array([9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0])   # MKZMPCPathFollower.jl:51-59
W_FRENET = np.array([9.0, 10.0, 0.5, 100.0, 1000.0, 0.0, 0.0])     # MKZMPCPathFollowerFrenet.jl:51-58


def weight_rows(B, n, seed):
    """Seeded rows log-uniform in [0.1x, 10x] the module defaults (entries whose default is 0 around 1 instead, so that every
    term of the cost is exercised), then one row of the defaults and one with zero input weights (ca = cd = 0)."""
    rng = np.random.default_rng(seed)
    base = (W_XY if n == 8 else W_FRENET).copy()
    scale = np.where(base > 0, base, 1.0)
    rows = scale * 10.0 ** rng.uniform(-1.0, 1.0, size=(B, n))
    rows[0] = base
    rows[1, -2:] = 0.0
    return rows


def xy_cfg(oracle, N, row):
    return oracle.default_cfg(N, weights=row)


def frenet_cfg(oracle, N, row):
    return oracle.default_cfg_frenet(N, weights=np.concatenate([[0.0], row]))


def oracle_per_row(oracle, make_cfg, solve, N, rows, *inputs):
    """The oracle, one problem at a time, each with its own weights."""
    outs = [solve(make_cfg(oracle, N, rows[b]), *[None if a is None else a[b:b + 1] for a in inputs]) for b in range(rows.shape[0])]
    return {k: np.concatenate([o[k] for o in outs]) for k in ("u0", "status", "iters", "cost")}


def check(o, e):
    assert (o["status"] == e["status"]).all()
    short = o["iters"] < 100
    assert (o["iters"][short] == e["iters"][short]).all()
    ok = o["status"] == 0
    assert ok.sum() >= len(ok) // 2
    assert np.abs(o["u0"] - e["u0"])[ok].max() <= 1e-9


@pytest.mark.parametrize("N,B,tpp", [(3, 24, False), (8, 24, False), (20, 12, False), (40, 4, False), (8, 32, True), (20, 16, True)])
def test_weighted_xy_matches_oracle(oracle, N, B, tpp):
    """Warp layout at N = 3, 8, 20 and 40 (a two-warp team), thread layout at N = 8 and 20."""
    import emu as E
    import emu_weights as EW
    b = W.make_batch(B, N)
    rows = weight_rows(B, 8, seed=N)
    o = oracle_per_row(oracle, xy_cfg, lambda c, *a: oracle.solve_batch(c, *a), N, rows, b["state"], b["ref"], b["v_des"], b["u_prev"])
    e = EW.solve_batch_w(E.kcfg_from_oracle(oracle.default_cfg(N)), b["state"], b["ref"], b["v_des"], b["u_prev"], rows, tpp=tpp, slots=7)
    check(o, e)


@pytest.mark.parametrize("N,B,tpp", [(8, 16, False), (20, 8, False), (8, 16, True), (20, 8, True)])
def test_weighted_frenet_matches_oracle(oracle, N, B, tpp):
    import emu as E
    import emu_weights as EW
    b = W.make_frenet_batch(B, N)
    rows = weight_rows(B, 7, seed=100 + N)
    o = oracle_per_row(oracle, frenet_cfg, lambda c, *a: oracle.solve_batch_frenet(c, *a), N, rows,
                       b["state"], b["kpoly"], b["v_des"], b["u_prev"])
    e = EW.solve_batch_frenet_w(E.kcfg_from_oracle(oracle.default_cfg_frenet(N)), b["state"], b["kpoly"], b["v_des"], b["u_prev"], rows,
                               tpp=tpp, slots=5)
    check(o, e)


@pytest.mark.parametrize("tpp", [False, True])
def test_mixed_batch_equals_unweighted_batches(oracle, tpp):
    """A batch mixing four weight vectors equals four unweighted batches, each with KCfg::w set to one of them."""
    import emu as E
    import emu_weights as EW
    N, B = 8, 32
    b = W.make_batch(B, N)
    vecs = weight_rows(4, 8, seed=7)
    which = np.arange(B) % 4
    k = E.kcfg_from_oracle(oracle.default_cfg(N))
    e = EW.solve_batch_w(k, b["state"], b["ref"], b["v_des"], b["u_prev"], vecs[which], tpp=tpp)
    for j in range(4):
        kj = E.kcfg_from_oracle(oracle.default_cfg(N, weights=vecs[j]))
        m = which == j
        fn = E.solve_batch_tpp if tpp else E.solve_batch
        u = fn(kj, b["state"][m], b["ref"][m], b["v_des"][m], b["u_prev"][m])
        assert (u["status"] == e["status"][m]).all() and (u["iters"] == e["iters"][m]).all()
        assert np.abs(u["u0"] - e["u0"][m]).max() <= 1e-12 and np.abs(u["cost"] - e["cost"][m]).max() <= 1e-12 * max(1.0, np.abs(u["cost"]).max())


@pytest.mark.parametrize("tpp", [False, True])
def test_weighted_rollout_matches_oracle_closed_loop(oracle, tpp):
    """The fused kernel's source and the per-period pipeline with per-vehicle weights, against the oracle's closed loop with each
    vehicle's own weights (the first solve of every vehicle still starts from the module-load solution of the default problem)."""
    import emu as E
    import emu_weights as EW
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    g = GPSRefTrajectory(mat_filename=1)
    N, T = 8, 10
    cfg = oracle.default_cfg(N)
    rng = np.random.default_rng(5)
    poses = np.array([g.trajectory[j, [4, 5, 3]] + rng.normal(scale=[0.3, 0.3, 0.03]) for j in (0, 900, 2500, 4000, 5200)])
    rows = weight_rows(poses.shape[0], 8, seed=11)
    seed = oracle.module_load_solution(cfg)
    log, final = EW.rollout_w(E.kcfg_from_oracle(cfg), g.trajectory, poses, T, rows, warm0=seed, tpp=tpp)
    path, keep = oracle.make_path(g.trajectory)
    for v in range(poses.shape[0]):
        olog = oracle.closed_loop(oracle.default_cfg(N, weights=rows[v]), path, poses[v], T)
        assert np.array_equal(log[:, v, 6], olog[:, 6]) and np.array_equal(log[:, v, 7], olog[:, 7]), v
        assert np.abs(log[:, v, 4:6] - olog[:, 4:6]).max() <= 1e-9, v
        assert np.abs(log[:, v, 0:4] - olog[:, 0:4]).max() <= 1e-9, v


@pytest.mark.parametrize("tpp", [False, True])
def test_bad_row_is_answered_with_error(oracle, tpp):
    """A negative or NaN weight (what device pointers cannot have checked on the host): MPCB200_ERROR and zero commands for that
    problem only; its neighbours are solved as without it."""
    import emu as E
    import emu_weights as EW
    N, B = 8, 6
    b = W.make_batch(B, N)
    rows = np.tile(W_XY, (B, 1))
    rows[1, 3] = -1.0
    rows[4, 6] = np.nan
    k = E.kcfg_from_oracle(oracle.default_cfg(N))
    e = EW.solve_batch_w(k, b["state"], b["ref"], b["v_des"], b["u_prev"], rows, tpp=tpp)
    u = (E.solve_batch_tpp if tpp else E.solve_batch)(k, b["state"], b["ref"], b["v_des"], b["u_prev"])
    bad = np.isin(np.arange(B), [1, 4])
    assert (e["status"][bad] == 4).all() and (e["u0"][bad] == 0).all() and (e["iters"][bad] == 0).all()
    assert (e["cost"][bad] == 0).all() and (e["n_resto"][bad] == 0).all()
    assert (e["status"][~bad] == u["status"][~bad]).all() and (e["iters"][~bad] == u["iters"][~bad]).all()
    assert np.array_equal(e["u0"][~bad], u["u0"][~bad])
