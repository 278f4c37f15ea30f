"""GPU tests of mpcb200_solve_batch_frenet_on_path through the C ABI: Frenet-frame batches from vehicle poses.

The call is on_path_frenet_ref_kernel (frenet_on_path_problem: the node's reference step from each pose into k_coeffs_out and
state_out), the solve kernel mpcb200_solve_batch_frenet would take for the same batch, and on_path_invalid_kernel.
1. k_coeffs_out / state_out against frenet_on_path_ref (np.argmin, np.interp, oracle.frenet_fit) for the pose classes of
   test_frenet_on_path_emu.py (on, beside, across the path, near its end, 2 km away), windows 4, 40, 40.3, 500, e_y from the path
   and e_y = 0.
2. u0, cost, status, iters, traj and warm bit-identical to solve_batch_frenet(_w) on the returned rows, in every layout:
   mpc_solve_frenet_kernel<4> and <3> (MPCB200_FRENET_WPB), the long teams (N = 40, 80), the thread-per-problem kernel
   (set_large_batch_path(1), and the default rule at 65,536 problems with N = 20); with and without weight rows, warm in and out.
3. Iterate for iterate against the oracle on the reference's rows at max_iter 1 and 3 and uncapped.
4. Device pointers give the host call's results bit for bit; an unset path id and a negative weight row give MPCB200_ERROR for
   that problem alone.  5. Rejected arguments.  6. Launch counts, restorations.  7. Two GPUs.
8. The node's loop with an external plant (oracle.plant_step), one call per period carrying warm and u_prev, against
   oracle.closed_loop_frenet.
Bars are 10x the largest difference measured on a B200 (1,000 W power limit), rounded up to one digit (measured values beside
them).  `pytest -s` prints the observed table."""
import contextlib
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from frenet_on_path_ref import batch3, far_poses, frenet_on_path_batch  # noqa: E402

pytestmark = pytest.mark.gpu

# 1. reference rows: K(s) on the 0.25 m grid relative to max |K|, psi_start absolute, e_y relative to max(1, |e_y|); poses near
#    the path / 2 km away (far_poses).  Measured: K near 6.85e-12 (w = 4), 1.47e-12 (40), 8.74e-13 (40.3), 1.30e-10 (500: the pose
#    near the end); K far 1.64e-9, 4.15e-11, 9.68e-12, 2.45e-14; psi_start 4.08e-15 / 2.19e-12; e_y 6.46e-16 / 8.67e-13
K_BAR = {"near": {4.0: 7e-11, 40.0: 2e-11, 40.3: 9e-12, 500.0: 2e-9}, "far": {4.0: 2e-8, 40.0: 5e-10, 40.3: 1e-10, 500.0: 3e-13}}
PSI_BAR = {"near": 5e-14, "far": 3e-11}
EY_BAR = {"near": 7e-15, "far": 9e-12}
# 3. capped iterates: traj relative to max(1, |x|); measured 5.74e-15 (N3), 3.63e-14 (N8), 3.78e-14 (N20), 2.67e-14 (N31),
#    3.63e-14 (tpp_N8)
ITER_BARS = {"N3": 6e-14, "N8": 4e-13, "N20": 4e-13, "N31": 3e-13, "tpp_N8": 4e-13}
#    uncapped: |du0|; measured 2.14e-15, 3.80e-13, 4.16e-17, 7.98e-17, 3.78e-13
FULL_BARS = {"N3": 3e-14, "N8": 4e-12, "N20": 5e-16, "N31": 8e-16, "tpp_N8": 4e-12}
# 8. the node's loop: poses and commands relative to max(1, |x|); measured 5.41e-16
LOOP_BAR = 6e-15

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


@contextlib.contextmanager
def frenet_wpb(wpb):
    """MPCB200_FRENET_WPB for the handles created inside (read when a handle is created)."""
    keep = os.environ.get("MPCB200_FRENET_WPB")
    if wpb is not None:
        os.environ["MPCB200_FRENET_WPB"] = str(wpb)
    try:
        yield
    finally:
        if keep is None:
            os.environ.pop("MPCB200_FRENET_WPB", None)
        else:
            os.environ["MPCB200_FRENET_WPB"] = keep


def solver(capi, tables, N, wpb=None, **kw):
    with frenet_wpb(wpb):
        s = capi.FrenetSolver(N, **kw)
    for p, tr in enumerate(tables):
        s.set_path(p, tr)
    return s


def fleet(tables, B, seed):
    """B poses (X, Y, psi, v) beside paths 0, 1, 2, 0, ... (0.4 m, 0.05 rad noise), spread along them; u_prev, v_des, weight rows."""
    rng = np.random.default_rng(seed)
    path_of = (np.arange(B) % 3).astype(np.int32)
    pose = np.empty((B, 4))
    for p in range(3):
        m = path_of == p
        tr = tables[p]
        idx = rng.integers(0, tr.shape[0] - 400, m.sum())
        pose[m, :3] = tr[idx][:, [4, 5, 3]] + rng.normal(scale=[0.4, 0.4, 0.05], size=(m.sum(), 3))
    pose[:, 3] = rng.uniform(2.0, 9.0, B)
    u_prev = rng.uniform(-0.05, 0.05, (B, 2))
    v_des = rng.uniform(6.0, 10.0, B)
    w = rng.uniform(0.5, 2.0, (B, 7)) * np.array([9.0, 10.0, 0.5, 100.0, 1000.0, 0.5, 0.5])
    return pose, path_of, u_prev, v_des, w


# ---- 1. reference rows
@pytest.mark.parametrize("window", [4.0, 40.0, 40.3, 500.0])
def test_reference_rows_match_oracle(capi, oracle, tables, window):
    s = solver(capi, tables, 8)
    pose, path_of = batch3(tables, window)
    B = pose.shape[0]
    g1 = s.solve_batch_on_path(pose, path_of, np.zeros((B, 2)), window=window, ey_from_path=True, want_ref=True)
    g0 = s.solve_batch_on_path(pose, path_of, np.zeros((B, 2)), window=window, ey_from_path=False, want_ref=True)
    assert np.array_equal(g0["k_coeffs"], g1["k_coeffs"]) and (g0["state"][:, 1] == 0.0).all()
    assert np.array_equal(g0["state"][:, [0, 2, 3]], g1["state"][:, [0, 2, 3]])
    K, S = frenet_on_path_batch(oracle, tables, pose, path_of, window, True)
    far = far_poses(tables, pose, path_of)
    grid = np.arange(0.0, window, 0.25)
    k, st = g1["k_coeffs"], g1["state"]
    assert (st[:, 0] == 0.0).all() and np.array_equal(st[:, 3], pose[:, 3])
    for b in range(B):
        c = "far" if far[b] else "near"
        Ke = np.polyval(K[b], grid)
        observe("K_w%g_%s" % (window, c), np.abs(np.polyval(k[b], grid) - Ke).max() / np.abs(Ke).max(), K_BAR[c][window])
        observe("psi_start_" + c, abs(st[b, 2] - S[b, 2]), PSI_BAR[c])
        observe("e_y_" + c, abs(st[b, 1] - S[b, 1]) / max(1.0, abs(S[b, 1])), EY_BAR[c])


# ---- 2. bit-identity with solve_batch_frenet(_w) on the returned rows
# id: (N, B, MPCB200_FRENET_WPB, large-batch threshold or None = default rule)
LAYOUTS = {
    "wpb4_N8": (8, 300, 4, 0),
    "wpb3_N8": (8, 300, 3, 0),
    "wpb4_N20": (20, 300, 4, 0),
    "long2_N40": (40, 200, None, 0),
    "long3_N80": (80, 100, None, 0),
    "tpp_N8": (8, 300, None, 1),
    "default_N20_65536": (20, 65536, None, None),
}
FIELDS = ("u0", "cost", "status", "iters", "traj")


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_bit_identical_to_solve_batch_frenet(capi, tables, layout):
    N, B, wpb, tpp = LAYOUTS[layout]
    s = solver(capi, tables, N, wpb=wpb)
    if tpp is not None:
        s.set_large_batch_path(tpp)
    pose, path_of, u_prev, v_des, w = fleet(tables, B, seed=N)
    warm0 = s.solve_batch_on_path(pose, path_of, u_prev, want_traj=True)["traj"]
    for weights in (None, w):
        for use_warm, vd in ((False, None), (True, v_des)):
            wa = warm0.copy() if use_warm else None
            g = s.solve_batch_on_path(pose, path_of, u_prev, v_des=vd, warm=wa, want_traj=True, want_ref=True, weights=weights)
            wb = warm0.copy() if use_warm else None
            o = s.solve_batch(g["state"], g["k_coeffs"], u_prev, v_des=np.full(B, 8.0) if vd is None else vd, warm=wb, want_traj=True,
                              weights=weights)
            for f in FIELDS:
                assert np.array_equal(g[f], o[f]), (layout, f, weights is None, use_warm)
            if use_warm:
                assert np.array_equal(wa, wb), (layout, "warm")
            assert (g["status"] == 0).mean() > 0.95, (layout, np.bincount(g["status"]))


# ---- 3. iterate for iterate against the oracle
ITER_ROWS = {"N3": (3, 0), "N8": (8, 0), "N20": (20, 0), "N31": (31, 0), "tpp_N8": (8, 1)}


@pytest.mark.parametrize("row", list(ITER_ROWS))
def test_iterates_match_oracle(capi, oracle, tables, row):
    N, tpp = ITER_ROWS[row]
    B = 12
    pose, path_of, u_prev, v_des, _ = fleet(tables, B, seed=100 + N)
    K, S = frenet_on_path_batch(oracle, tables, pose, path_of, 40.0, True)
    for max_iter in (1, 3, None):
        kw = {} if max_iter is None else {"max_iter": max_iter}
        s = solver(capi, tables, N, **kw)
        s.set_large_batch_path(tpp)
        g = s.solve_batch_on_path(pose, path_of, u_prev, v_des=v_des, want_traj=True)
        cfg = oracle.default_cfg_frenet(N, max_iter=s.cfg.max_iter)
        o = oracle.solve_batch_frenet(cfg, S, K, v_des, u_prev, want_traj=True)
        assert np.array_equal(g["status"], o["status"]), (row, max_iter, g["status"], o["status"])
        assert np.array_equal(g["iters"], o["iters"]), (row, max_iter, g["iters"], o["iters"])
        if max_iter is not None:
            assert (o["status"] == 3).all()
            observe("iter_" + row, (np.abs(g["traj"] - o["traj"]) / np.maximum(1.0, np.abs(o["traj"]))).max(), ITER_BARS[row])
        else:
            assert (o["status"] == 0).all()
            observe("full_" + row, np.abs(g["u0"] - o["u0"]).max(), FULL_BARS[row])


# ---- 4. device pointers
def test_device_pointers(capi, tables):
    import torch
    N, B = 8, 257
    s = solver(capi, tables, N)
    pose, path_of, u_prev, v_des, w = fleet(tables, B, seed=5)
    h = s.solve_batch_on_path(pose, path_of, u_prev, want_traj=True, want_ref=True, weights=w)
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    def run(pof, wr):
        out = {"u0": torch.empty((B, 2), dtype=torch.float64, device=dev), "cost": torch.empty(B, dtype=torch.float64, device=dev),
               "status": torch.empty(B, dtype=torch.int32, device=dev), "iters": torch.empty(B, dtype=torch.int32, device=dev),
               "traj": torch.empty((B, 6 * N + 4), dtype=torch.float64, device=dev),
               "k_coeffs": torch.empty((B, 4), dtype=torch.float64, device=dev), "state": torch.empty((B, 4), dtype=torch.float64, device=dev)}
        s.solve_batch_on_path_device(B, t(pose), t(pof), t(u_prev), out["u0"], cost=out["cost"], status=out["status"], iters=out["iters"],
                                     traj=out["traj"], k_coeffs_out=out["k_coeffs"], state_out=out["state"], weights=t(wr))
        torch.cuda.synchronize()
        return {k: v.cpu().numpy() for k, v in out.items()}

    d = run(path_of, w)
    for f in FIELDS + ("k_coeffs", "state"):
        assert np.array_equal(d[f], h[f]), f
    assert s.stats()["kernel_launches"] == 3
    bad_path, bad_w = np.array([3, 100]), np.array([7, 200])
    pof = path_of.copy(); pof[bad_path[0]] = -1; pof[bad_path[1]] = 5
    wr = w.copy(); wr[bad_w[0], 2] = -1.0; wr[bad_w[1], 6] = np.nan
    d = run(pof, wr)
    bad = np.zeros(B, dtype=bool); bad[bad_path] = True; bad[bad_w] = True
    assert (d["status"][bad] == capi.ERROR).all() and (d["u0"][bad] == 0).all() and (d["cost"][bad] == 0).all() and (d["iters"][bad] == 0).all()
    assert np.isnan(d["k_coeffs"][bad_path]).all() and np.isnan(d["state"][bad_path]).all()
    assert np.array_equal(d["k_coeffs"][bad_w], h["k_coeffs"][bad_w])
    for f in FIELDS + ("k_coeffs", "state"):
        assert np.array_equal(d[f][~bad], h[f][~bad]), f


# ---- 5. rejected arguments
def test_rejected_arguments(capi, tables):
    N, B = 8, 4
    s = solver(capi, tables, N)
    s.close()
    s = capi.FrenetSolver(N)
    s.set_path(0, tables[0])
    pose, path_of, u_prev, v_des, w = fleet(tables, B, seed=9)
    path_of[:] = 0
    L = capi.lib()
    u0 = np.empty((B, 2))
    p = lambda a: None if a is None else a.ctypes.data

    def call(h, pose_=pose, pof=path_of, window=40.0, up=u_prev, u0_=u0, w_=None):
        return L.mpcb200_solve_batch_frenet_on_path(h, B, p(pose_), p(pof), window, 8.0, 1, None, p(up), None, p(w_), p(u0_),
                                                     None, None, None, None, None, None, capi.HOST)

    name = b"mpcb200_solve_batch_frenet_on_path"
    xy = capi.Solver(N)
    assert call(xy._h) == -1 and name in L.mpcb200_last_error(xy._h)
    assert b"mpcb200_create_frenet" in L.mpcb200_last_error(xy._h)
    cases = [dict(window=3.9), dict(window=500.1), dict(window=float("nan")), dict(pof=np.array([0, 1, 0, 0], dtype=np.int32)),
             dict(pose_=None), dict(pof=None), dict(up=None), dict(u0_=None), dict(w_=np.where(np.arange(7) == 3, -1.0, w))]
    for kw in cases:
        assert call(s._h, **kw) == -1, kw
        assert name in L.mpcb200_last_error(s._h), (kw, L.mpcb200_last_error(s._h))
    call(s._h, pof=np.array([0, 1, 0, 0], dtype=np.int32))
    assert b"problem 1 uses path 1" in L.mpcb200_last_error(s._h)
    call(s._h, w_=np.where(np.arange(7) == 3, -1.0, w))
    assert b"weight 3 of problem 0" in L.mpcb200_last_error(s._h)
    assert call(s._h) == 0 and (np.isfinite(u0)).all()
    assert L.mpcb200_solve_batch_on_path(s._h, B, p(pose), p(path_of), 1, 8.0, None, p(u_prev), None, p(u0), None, None, None, None,
                                         None, None, capi.HOST) == -1


# ---- 6. launches and restorations
def test_launches_and_restorations(capi, tables):
    s = solver(capi, tables, 8)
    for B in (1, 100, 5000):
        pose, path_of, u_prev, _, _ = fleet(tables, B, seed=B)
        g = s.solve_batch_on_path(pose, path_of, u_prev)
        assert s.stats()["kernel_launches"] == 3 and s.stats()["kernel_ms"] > 0
        r = s.restorations(B)
        assert r.shape == (B,) and (r >= 0).all() and (g["status"] == 0).mean() > 0.95


# ---- 7. two GPUs
def test_two_gpus_equal_one(capi, tables):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    N, B = 8, 500
    one, two = solver(capi, tables, N), solver(capi, tables, N, devices=[0, 1])
    pose, path_of, u_prev, v_des, w = fleet(tables, B, seed=7)
    for weights in (None, w):
        a = one.solve_batch_on_path(pose, path_of, u_prev, v_des=v_des, want_traj=True, want_ref=True, weights=weights)
        b = two.solve_batch_on_path(pose, path_of, u_prev, v_des=v_des, want_traj=True, want_ref=True, weights=weights)
        for f in FIELDS + ("k_coeffs", "state"):
            assert np.array_equal(a[f], b[f]), f
        assert (two.restorations(B) >= 0).all()


# ---- 8. the node's loop around an external plant
def test_node_loop_with_external_plant(capi, oracle, tables):
    """40 periods: oracle.plant_step drives each vehicle (ten publishes per period), one call per period carries warm and u_prev
    (update_current_input(df, acc)); against oracle.closed_loop_frenet vehicle by vehicle."""
    N, T, window = 8, 40, 40.0
    s = solver(capi, tables, N)
    rng = np.random.default_rng(3)
    path_of = np.array([0, 1, 2], dtype=np.int32)
    pose0 = np.array([tables[p][[600, 2100, 3500][p], [4, 5, 3]] + rng.normal(scale=[0.3, 0.3, 0.03]) for p in path_of])
    B = 3
    st = np.zeros((B, 8)); st[:, :3] = pose0
    acc = np.zeros(B); df = np.zeros(B)
    u_prev = np.zeros((B, 2)); warm = np.zeros((B, 6 * N + 4)); log = np.zeros((T, B, 8))
    for t in range(T):
        for b in range(B):
            for _ in range(10):
                st[b] = oracle.plant_step(st[b], acc[b], df[b])
        g = s.solve_batch_on_path(st[:, :4], path_of, u_prev, window=window, target_vel=8.0, warm=warm)
        acc, df = g["u0"][:, 0].copy(), g["u0"][:, 1].copy()
        u_prev[:, 0] = df; u_prev[:, 1] = acc
        log[t] = np.column_stack([st[:, :4], acc, df, g["status"], g["iters"]])
    cfg = oracle.default_cfg_frenet(N)
    olog = np.stack([oracle.closed_loop_frenet(cfg, tables[p], pose0[b], T, window, 8.0, True) for b, p in enumerate(path_of)], axis=1)
    assert np.array_equal(log[:, :, 6], olog[:, :, 6]) and (olog[:, :, 6] == 0).mean() >= 0.9
    assert np.abs(log[:, :, 7] - olog[:, :, 7]).max() <= 1
    observe("node_loop", (np.abs(log[:, :, :6] - olog[:, :, :6]) / np.maximum(1.0, np.abs(olog[:, :, :6]))).max(), LOOP_BAR)
