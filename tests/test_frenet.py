"""Frenet-frame variant (scripts/mpc_utils/MKZMPCPathFollowerFrenet.jl, SURVEY.md 8 f-3): oracle NLP restatement
(finite-difference checks of the analytic derivatives), the curvature-polynomial fit of
scripts/sim_path_utils/nav_msgs_path_frenet.py, and the CUDA solver's source on the CPU warp emulator against
the oracle, iterate for iterate.  The -m gpu tests of the same path are in test_gpu_parity.py."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from mkz_mpc_path_follower_b200 import frenet_ref, workload as W

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))


def _p(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


@pytest.mark.parametrize("N", [4, 7])
def test_frenet_derivatives_fd(oracle, N):
    """Jacobian and Lagrangian Hessian of the Frenet stage map (:111-120) against central differences."""
    rng = np.random.default_rng(11)
    cfg = oracle.default_cfg_frenet(N, weights=[0, 9, 10, 0.5, 100, 1000, 0.3, 0.7])
    for i, v in enumerate([2e-5, -3e-4, 2e-3, 0.02]):
        cfg.kpoly[i] = v
    L = oracle.lib()
    n, mc, md = 6 * N + 4, 4 * N + 4, 2 * (N - 1)
    z = rng.normal(size=n)
    for k in range(N + 1):
        z[6 * k:6 * k + 4] = [rng.uniform(0, 20), rng.uniform(-1, 1), rng.uniform(-0.5, 0.5), rng.uniform(0.5, 15)]
        if k < N:
            z[6 * k + 4:6 * k + 6] = [rng.uniform(-1, 1), rng.uniform(-0.5, 0.5)]
    state = rng.normal(size=4); yc = rng.normal(size=mc)

    def c(zz):
        o = np.empty(mc); L.mpc_oracle_eval_c(C.byref(cfg), _p(state), _p(zz), _p(o)); return o

    def jac(zz):
        J1 = np.empty((mc, n)); J2 = np.empty((md, n)); L.mpc_oracle_eval_jac(C.byref(cfg), _p(zz), _p(J1), _p(J2)); return J1

    H = np.empty((n, n)); L.mpc_oracle_eval_hess(C.byref(cfg), _p(z), 0.0, _p(yc), _p(H))
    J = jac(z); h = 1e-6
    Jfd = np.empty((mc, n)); Hfd = np.empty((n, n))
    for i in range(n):
        e = np.zeros(n); e[i] = h
        Jfd[:, i] = (c(z + e) - c(z - e)) / (2 * h)
        Hfd[:, i] = (jac(z + e).T @ yc - jac(z - e).T @ yc) / (2 * h)
    assert np.abs(J - Jfd).max() <= 1e-7
    assert np.abs(H - Hfd).max() <= 1e-7 and np.abs(H - H.T).max() == 0.0
    assert np.abs(H).max() > 0.1    # the test is not vacuous
    # the stage map itself, against the formulas of the reference written out in numpy
    k0, k1, k2, k3 = (cfg.kpoly[i] for i in range(4))
    s, ey, ep, v, a, d = z[0:6]
    K = k0 * s ** 3 + k1 * s ** 2 + k2 * s + k3
    bta = np.arctan(cfg.L_b / (cfg.L_a + cfg.L_b) * np.tan(d))
    dsdt = v * np.cos(ep + bta) / (1 - ey * K)
    nxt = np.array([s + 0.2 * dsdt, ey + 0.2 * v * np.sin(ep + bta), ep + 0.2 * (v / cfg.L_b * np.sin(bta) - dsdt * K), v + 0.2 * a])
    assert np.abs((z[6:10] - nxt) - c(z)[4:8]).max() <= 1e-13


def test_frenet_reference_fit():
    """get_reference_frenet (nav_msgs_path_frenet.py:76-86): an arc of radius 100 m gives K = 1/100 (a cubic X(s), Y(s) cannot follow much tighter arcs over 40 m) and the
    start heading; the batched form used by the workload is the same arithmetic."""
    R, th0 = 100.0, 0.3
    s = np.arange(0.0, 40.0, 0.8)
    x = R * (np.sin(th0 + s / R) - np.sin(th0)); y = -R * (np.cos(th0 + s / R) - np.cos(th0))
    K, psi0, xi, yi = frenet_ref.get_reference_frenet({"x": x, "y": y, "s": s})
    sq = np.linspace(0, 35, 8)
    assert np.abs(np.polyval(K, sq) - 1.0 / R).max() <= 5e-4
    assert abs(psi0 - th0) <= 0.02
    s_fit = np.arange(0.0, s[-1], 0.5)
    Kb, pb = frenet_ref.fit_windows(np.interp(s_fit, s, x)[None], np.interp(s_fit, s, y)[None], s[-1])
    assert np.allclose(Kb[0], K, rtol=1e-9, atol=1e-12) and abs(pb[0] - psi0) <= 1e-12


def _stress_batch(B, N, seed):
    """Tighter curves and larger offsets than the recorded paths give: K up to ~0.05 1/m varying along s."""
    rng = np.random.default_rng(seed)
    b = W.make_frenet_batch(B, N)
    b["kpoly"] = np.stack([rng.uniform(-2e-6, 2e-6, B), rng.uniform(-1e-4, 1e-4, B), rng.uniform(-2e-3, 2e-3, B),
                           rng.uniform(-0.05, 0.05, B)], axis=1)
    b["state"][:, 1] = rng.uniform(-1.0, 1.0, B)
    b["state"][:, 2] = rng.uniform(-0.3, 0.3, B)
    return b


@pytest.mark.parametrize("N,B,stress", [(8, 16, False), (20, 10, False), (3, 6, False), (31, 3, False), (8, 12, True), (20, 8, True),
                                            (32, 2, False), (40, 3, True), (64, 2, False), (80, 2, True)])
def test_emulated_frenet_kernel_matches_oracle(oracle, N, B, stress):
    import emu as E
    E.race_check(True)
    cfg = oracle.default_cfg_frenet(N)
    b = _stress_batch(B, N, 5) if stress else W.make_frenet_batch(B, N)
    o = oracle.solve_batch_frenet(cfg, b["state"], b["kpoly"], b["v_des"], b["u_prev"], want_traj=True, n_threads=4)
    e = E.solve_batch_frenet(E.kcfg_from_oracle(cfg), b["state"], b["kpoly"], b["v_des"], b["u_prev"], want_traj=True)
    assert E.race_count() == 0
    assert (o["status"] == e["status"]).all() and (o["iters"] == e["iters"]).all()
    ok = o["status"] == 0
    assert ok.sum() >= B - 1
    assert np.abs(o["u0"] - e["u0"])[ok].max() <= 1e-9
    assert (np.abs(o["cost"] - e["cost"])[ok] <= 1e-9 * np.maximum(1, np.abs(o["cost"][ok]))).all()
    assert np.abs(o["traj"] - e["traj"])[ok].max() <= 1e-8
    # warm start from the solution: a handful of iterations, same point
    wo, we = o["traj"].copy(), o["traj"].copy()
    o2 = oracle.solve_batch_frenet(cfg, b["state"], b["kpoly"], b["v_des"], b["u_prev"], warm=wo, n_threads=4)
    e2 = E.solve_batch_frenet(E.kcfg_from_oracle(cfg), b["state"], b["kpoly"], b["v_des"], b["u_prev"], warm=we)
    assert (o2["status"] == e2["status"]).all() and (o2["iters"] == e2["iters"]).all()
    assert np.abs(o2["u0"] - e2["u0"])[o2["status"] == 0].max() <= 1e-9
    assert np.abs(o2["u0"] - o["u0"])[ok & (o2["status"] == 0)].max() <= 1e-6


def test_emulated_frenet_rollout_start(oracle):
    """MPCB200_START_ROLLOUT for the Frenet variant: the rollout uses the Frenet stage map."""
    import emu as E
    N, B = 8, 6
    cfg = oracle.default_cfg_frenet(N)
    b = _stress_batch(B, N, 9)
    e = E.solve_batch_frenet(E.kcfg_from_oracle(cfg, start_mode=1), b["state"], b["kpoly"], b["v_des"], b["u_prev"])
    o = oracle.solve_batch_frenet(cfg, b["state"], b["kpoly"], b["v_des"], b["u_prev"], n_threads=4)
    both = (o["status"] == 0) & (e["status"] == 0)
    assert both.sum() >= B - 1
    assert np.abs(o["u0"] - e["u0"])[both].max() <= 1e-5   # two start points, one optimum


def frenet_kkt_check(oracle, cfg, b, traj, status):
    """KKT conditions of the unscaled Frenet NLP at returned points (no interior-point code involved): equality rows
    satisfied, and the objective gradient lies in the span of the gradients of the equality rows and of the active
    rate rows / bounds."""
    N = cfg.N
    L = oracle.lib()
    n, mc, md = 6 * N + 4, 4 * N + 4, 2 * (N - 1)
    zero_ref = np.zeros(3 * (N + 1))
    checked = 0
    for j in np.nonzero(status == 0)[0]:
        for i in range(4):
            cfg.kpoly[i] = b["kpoly"][j, i]
        z = np.empty(n); L.mpc_oracle_traj_to_z(C.byref(cfg), _p(np.ascontiguousarray(traj[j])), _p(z))
        cv = np.empty(mc); L.mpc_oracle_eval_c(C.byref(cfg), _p(np.ascontiguousarray(b["state"][j])), _p(z), _p(cv))
        assert np.abs(cv).max() <= 1e-7
        g = np.empty(n); L.mpc_oracle_eval_grad_f(C.byref(cfg), _p(zero_ref), float(b["v_des"][j]), _p(z), _p(g))
        Jc = np.empty((mc, n)); Jd = np.empty((md, n)); L.mpc_oracle_eval_jac(C.byref(cfg), _p(z), _p(Jc), _p(Jd))
        d = np.empty(md); L.mpc_oracle_eval_d(C.byref(cfg), _p(np.ascontiguousarray(b["u_prev"][j])), _p(z), _p(d))
        lim = np.array([(cfg.steer_dmax if r % 2 == 0 else cfg.a_dmax) * (cfg.dt_control if r < 2 else cfg.dt) for r in range(md)])
        assert (np.abs(d) <= lim + 1e-7).all()
        lo = np.full(n, -np.inf); hi = np.full(n, np.inf)
        for k in range(N + 1):
            lo[6 * k + 3], hi[6 * k + 3] = cfg.v_min, cfg.v_max
            if k < N:
                lo[6 * k + 4], hi[6 * k + 4] = -cfg.a_max, cfg.a_max
                lo[6 * k + 5], hi[6 * k + 5] = -cfg.steer_max, cfg.steer_max
        assert (z >= lo - 1e-9).all() and (z <= hi + 1e-9).all()
        # multipliers: free for the equality rows, >= 0 for every inequality within 1e-3 of its limit (an interior-point
        # solution leaves weakly active constraints a slack of mu / multiplier); non-negative least squares on
        #   g + Jc' y + sum_i m_i n_i = 0,   n_i = outward normal of inequality i
        normals, slacks = [], []
        for r in range(md):
            for sgn in (1.0, -1.0):
                sl = lim[r] - sgn * d[r]
                if sl <= 1e-3:
                    normals.append(sgn * Jd[r]); slacks.append(max(sl, 0.0))
        eye = np.eye(n)
        for i in range(n):
            if hi[i] - z[i] <= 1e-3:
                normals.append(eye[i]); slacks.append(max(hi[i] - z[i], 0.0))
            if z[i] - lo[i] <= 1e-3:
                normals.append(-eye[i]); slacks.append(max(z[i] - lo[i], 0.0))
        cols = [Jc.T, -Jc.T] + ([np.array(normals).T] if normals else [])
        from scipy.optimize import nnls
        mult, _ = nnls(np.hstack(cols), -g, maxiter=20000)
        resid = g + np.hstack(cols) @ mult
        assert np.abs(resid).max() <= 1e-5 * max(1.0, np.abs(g).max())
        if normals:   # complementarity
            assert (mult[2 * mc:] * np.array(slacks)).max() <= 1e-5
        checked += 1
    return checked


def test_frenet_kkt_of_oracle_solutions(oracle):
    """The returned points satisfy the KKT conditions of the unscaled Frenet NLP (intrinsic check; parity unpinned)."""
    N, B = 8, 12
    cfg = oracle.default_cfg_frenet(N)
    b = _stress_batch(B, N, 3)
    o = oracle.solve_batch_frenet(cfg, b["state"], b["kpoly"], b["v_des"], b["u_prev"], want_traj=True, n_threads=4)
    assert frenet_kkt_check(oracle, cfg, b, o["traj"], o["status"]) >= B - 1


def frenet_edge_batch(N):
    """NaN curvature; 1 - e_y K = 0 at the start (the reference's ds/dt is singular there, :113); 1 - e_y K < 0;
    v0 above v_max (the only way this NLP is infeasible); a large s0; an ordinary problem."""
    b = W.make_frenet_batch(6, N)
    b["kpoly"][0, :] = np.nan
    b["kpoly"][1, :] = [0, 0, 0, 1.0]; b["state"][1, 1] = 1.0
    b["kpoly"][2, :] = [0, 0, 0, 0.5]; b["state"][2, 1] = 2.5
    b["state"][3, 3] = 25.0
    b["state"][4, :] = [1e3, 0.1, 0.0, 5.0]
    return b


def test_emulated_frenet_edge_cases(oracle):
    """Degenerate inputs end with the oracle's status and iteration count -- no hang, no divergence between the two."""
    import emu as E
    N = 8
    b = frenet_edge_batch(N)
    cfg = oracle.default_cfg_frenet(N, max_iter=60)
    o = oracle.solve_batch_frenet(cfg, b["state"], b["kpoly"], b["v_des"], b["u_prev"], n_threads=1)
    e = E.solve_batch_frenet(E.kcfg_from_oracle(cfg), b["state"], b["kpoly"], b["v_des"], b["u_prev"])
    assert o["status"].tolist() == [4, 4, 3, 1, 0, 0]
    assert (o["status"] == e["status"]).all() and (o["iters"] == e["iters"]).all()
    ok = o["status"] == 0
    assert np.abs(o["u0"] - e["u0"])[ok].max() <= 1e-9


def test_frenet_agrees_with_scipy_slsqp(oracle):
    """Independent solver on an independent transcription: scipy SLSQP minimises the Frenet NLP whose objective and
    constraint VALUES are written here in numpy straight from MKZMPCPathFollowerFrenet.jl:75-123 (derivatives from the
    oracle's analytic Jacobians, which the finite-difference test above pins).  Started near the oracle's point it must
    stay there: same cost to 1e-6 relative, same first move to 1e-4 (SLSQP's own accuracy)."""
    from scipy.optimize import minimize
    from test_oracle_solver import _nlp
    N, B = 8, 6
    cfg = oracle.default_cfg_frenet(N)
    b = _stress_batch(B, N, 41)
    o = oracle.solve_batch_frenet(cfg, b["state"], b["kpoly"], b["v_des"], b["u_prev"], want_traj=True, n_threads=4)
    L = oracle.lib()
    La, Lb, dt = cfg.L_a, cfg.L_b, cfg.dt
    rng = np.random.default_rng(1)
    checked = 0
    for j in np.nonzero(o["status"] == 0)[0]:
        kp = b["kpoly"][j]; st = b["state"][j]; vt = float(b["v_des"][j])
        for i in range(4):
            cfg.kpoly[i] = kp[i]
        _, g_or, _, d, jac, lo, hi, dlim = _nlp(oracle, cfg, np.ascontiguousarray(st), np.zeros(3 * (N + 1)), vt, np.ascontiguousarray(b["u_prev"][j]))

        def unpack(z):
            Z = np.concatenate([z, [0.0, 0.0]]).reshape(N + 1, 6)
            return Z[:, 0], Z[:, 1], Z[:, 2], Z[:, 3], Z[:N, 4], Z[:N, 5]      # s, ey, epsi, v, acc, df

        def f(z):   # :95-101 (1-based i = 2..N+1 -> 0-based 1..N; speed term i = 2..N)
            s, ey, ep, v, acc, df = unpack(z)
            return (9.0 * (ey[1:] ** 2).sum() + 10.0 * (ep[1:] ** 2).sum() + 0.5 * ((v[1:N] - vt) ** 2).sum()
                    + 100.0 * (np.diff(acc) ** 2).sum() + 1000.0 * (np.diff(df) ** 2).sum())

        def c(z):   # :106-120
            s, ey, ep, v, acc, df = unpack(z)
            K = kp[0] * s[:N] ** 3 + kp[1] * s[:N] ** 2 + kp[2] * s[:N] + kp[3]
            bta = np.arctan(Lb / (La + Lb) * np.tan(df))
            dsdt = v[:N] * np.cos(ep[:N] + bta) / (1 - ey[:N] * K)
            rows = [np.array([s[0], ey[0], ep[0], v[0]]) - st]
            nxt = np.stack([s[:N] + dt * dsdt, ey[:N] + dt * (v[:N] * np.sin(ep[:N] + bta)),
                            ep[:N] + dt * (v[:N] / Lb * np.sin(bta) - dsdt * K), v[:N] + dt * acc], axis=1)
            cur = np.stack([s[1:], ey[1:], ep[1:], v[1:]], axis=1)
            return np.concatenate([rows[0], (cur - nxt).reshape(-1)])

        z0 = np.empty(6 * N + 4)
        L.mpc_oracle_traj_to_z(C.byref(cfg), _p(np.ascontiguousarray(o["traj"][j])), _p(z0))
        assert abs(f(z0) - o["cost"][j]) <= 1e-9 * max(1.0, o["cost"][j])       # the two transcriptions agree on the objective
        assert np.abs(c(z0)).max() <= 1e-7                                      # ... and on the dynamics
        cons = [{"type": "eq", "fun": c, "jac": lambda z: jac(z)[0]},
                {"type": "ineq", "fun": lambda z: dlim - d(z), "jac": lambda z: -jac(z)[1]},
                {"type": "ineq", "fun": lambda z: dlim + d(z), "jac": lambda z: jac(z)[1]}]
        res = minimize(f, z0 + 1e-2 * rng.normal(size=z0.size), jac=g_or, bounds=list(zip(lo, hi)), constraints=cons,
                       method="SLSQP", options={"ftol": 1e-15, "maxiter": 500})
        assert np.abs(c(res.x)).max() < 1e-7
        assert abs(res.fun - o["cost"][j]) <= 1e-6 * max(1.0, abs(o["cost"][j])), (j, res.fun, o["cost"][j])
        assert np.abs(res.x[4:6] - o["u0"][j]).max() < 1e-4, (j, res.x[4:6], o["u0"][j])
        checked += 1
    assert checked >= 4


def test_emulated_frenet_kernel_property(oracle):
    """Property-based: for random curvature polynomials, offsets, speeds, previous commands and target speeds the
    emulated CUDA source and the oracle end with the same status, and where that is Optimal with the same command."""
    import emu as E
    from hypothesis import given, settings, strategies as st
    N = 5
    cfg = oracle.default_cfg_frenet(N, max_iter=80)
    kc = E.kcfg_from_oracle(cfg)
    fl = lambda lo, hi: st.floats(min_value=lo, max_value=hi, allow_nan=False, allow_infinity=False)

    @settings(max_examples=30, deadline=None, derandomize=True)
    @given(fl(-2e-6, 2e-6), fl(-1e-4, 1e-4), fl(-3e-3, 3e-3), fl(-0.06, 0.06), fl(-1.5, 1.5), fl(-0.4, 0.4), fl(0.0, 20.0),
           fl(-0.5, 0.5), fl(-1.0, 1.0), fl(0.0, 15.0))
    def check(k0, k1, k2, k3, ey, ep, v, df0, a0, vt):
        state = np.array([[0.0, ey, ep, v]]); kp = np.array([[k0, k1, k2, k3]]); up = np.array([[df0, a0]]); vd = np.array([vt])
        o = oracle.solve_batch_frenet(cfg, state, kp, vd, up, n_threads=1)
        e = E.solve_batch_frenet(kc, state, kp, vd, up)
        assert o["status"][0] == e["status"][0]
        if o["status"][0] == 0:
            assert abs(int(o["iters"][0]) - int(e["iters"][0])) <= 1
            assert np.abs(o["u0"] - e["u0"]).max() <= 1e-7

    check()


def test_emulated_frenet_closed_loop(oracle):
    """rollout_group_frenet (mpcb200_rollout_frenet's kernel source) on the emulator: the path ahead, the two cubic
    least-squares fits of nav_msgs_path_frenet.py:44-86 as fixed matrices, state (0, e_y, -psi_start, v), warm-started
    solve, command feedback -- against oracle.closed_loop_frenet (np.polyfit fits, oracle solves, the oracle's plant).
    test_frenet_closed_loop_emu.py runs it iterate for iterate at more horizons, windows and fleets."""
    import emu as E
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    N, T, window, vt = 8, 6, 40.0, 8.0
    g = GPSRefTrajectory(mat_filename=1)
    cfg = oracle.default_cfg_frenet(N)
    rng = np.random.default_rng(8)
    poses = np.array([g.trajectory[j, [4, 5, 3]] + rng.normal(scale=[0.4, 0.4, 0.05]) for j in (300, 2500, 3900, 50, 1200)])
    log, final = E.rollout_frenet(E.kcfg_from_oracle(cfg), g.trajectory, poses, T, window=window, target_vel=vt)
    assert E.race_count() == 0
    for b in range(poses.shape[0]):
        h = oracle.closed_loop_frenet(cfg, g.trajectory, poses[b], T, window, vt)
        assert np.array_equal(log[:, b, 6], h[:, 6]) and (log[:, b, 6] == 0).all(), b
        assert np.abs(log[:, b, 7] - h[:, 7]).max() <= 1, b
        assert np.abs(log[:, b, 4:6] - h[:, 4:6]).max() <= 1e-6, (b, np.abs(log[:, b, 4:6] - h[:, 4:6]).max())
        assert np.abs(log[:, b, 0:4] - h[:, 0:4]).max() <= 1e-7, b
