"""The Frenet closed loop of the kernel sources (compiled for the host, tests/emu) against references that share nothing with them.

The fused kernel (rollout_group_frenet) and the per-period pipeline (rollout_frenet_ref_kernel, then
rollout_solve_tpp_kernel<1, 0>) fit the path ahead with fixed pseudo-inverse matrices and solve with the library's interior-point
code.  Here they are checked piece by piece:

  * fit grid sizes: fit_grid_sizes must give np.arange(0, window, 0.5).size and np.arange(0, window, 0.25).size, the grids of
    nav_msgs_path_frenet.py:63,79, for windows on and just off a multiple of the step;
  * fit matrices: cubic_fit_matrix against (V'V)^-1 V' in exact rational arithmetic (the grid points are multiples of 0.25);
  * frenet_reference: K(s), psi_start and e_y of one control period against the same chain computed exactly (fractions.Fraction)
    from the kernel's own samples of the path ahead, for poses on, beside and across the path, near its end, and windows of 4 to
    500 m;
  * the closed loop, iterate for iterate: both forms against oracle.closed_loop_frenet (np.polyfit fits, oracle solves, the
    oracle's plant) at max_iter = 1 and 3, where every period stops at an interior iterate, and uncapped.
A vehicle whose whole window lies past the path end is not compared: every sample is then the last point and K is 0/0.
`pytest -s` prints the largest difference seen per check next to its bar."""
import math
import os
import sys
from fractions import Fraction

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

WINDOWS = (4.0, 4.1, 40.0, 40.0 + 1e-10, 40.3, 123.75, 500.0 - 1e-10, 500.0)

# bars: 10x the largest difference measured with the host build (g++ -O1, no contraction), rounded up to one digit
FIT_MATRIX_BAR = 2e-14            # relative to each row's largest entry; measured 1.22e-15 (n = 2000); numpy's pinv: 9.2e-14
K_BAR = {4.0: 5e-11, 40.0: 9e-12, 40.3: 3e-11, 500.0: 2e-9}   # K(s) on the 0.25 m grid, relative to max |K|; measured
#                                 4.29e-12, 8.56e-13, 2.23e-12, 1.07e-10 (the largest are poses whose window straddles the path
#                                 end, where most samples are the last point and max |K| is small)
PSI_BAR = 8e-15                   # psi_start, absolute; measured 7.77e-16
EY_BAR = 9e-15                    # e_y, absolute; measured 8.88e-16
ITER_BAR = 1e-10                  # capped closed loop: poses and commands relative to max(1, |x|) (the bar of the iterate tests)
U_BAR = 1e-8                      # uncapped closed loop: commands

OBSERVED = {}


def observe(name, d, bar):
    OBSERVED[name] = (max(OBSERVED.get(name, (0.0, bar))[0], float(d)), bar)
    assert d <= bar, (name, d, bar)


@pytest.fixture(scope="module", autouse=True)
def _print_observed():
    yield
    for name in sorted(OBSERVED):
        print("observed %-28s %.2e  (bar %.0e)" % (name, OBSERVED[name][0], OBSERVED[name][1]))


@pytest.fixture(scope="module")
def tables():
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    return [GPSRefTrajectory(mat_filename=p).trajectory for p in (1, 2, 3)]


@pytest.fixture(autouse=True)
def _race_check():
    import emu as E
    E.race_check(True)
    yield
    assert E.race_count() == 0


# ---- exact arithmetic
def exact_fit_matrix(n, step):
    """(V'V)^-1 and V for the cubic least-squares fit on g * step, g < n, as Fractions (V rows: x^3, x^2, x, 1)."""
    xs = [Fraction(step) * g for g in range(n)]
    V = [[x ** (3 - c) for c in range(4)] for x in xs]
    A = [[sum(V[g][a] * V[g][b] for g in range(n)) for b in range(4)] + [Fraction(int(a == b)) for b in range(4)] for a in range(4)]
    for c in range(4):   # Gauss-Jordan on the SPD normal matrix (no pivoting needed in exact arithmetic)
        A[c] = [v / A[c][c] for v in A[c]]
        for r in range(4):
            if r != c:
                A[r] = [A[r][b] - A[r][c] * A[c][b] for b in range(8)]
    return [row[4:] for row in A], V


_EXACT = {}


def exact_fit(n, step):
    if (n, step) not in _EXACT:
        _EXACT[(n, step)] = exact_fit_matrix(n, step)
    return _EXACT[(n, step)]


def lsq_cubic(n, step, y):
    Gi, V = exact_fit(n, step)
    Vy = [sum(V[g][b] * y[g] for g in range(n)) for b in range(4)]
    return [sum(Gi[a][b] * Vy[b] for b in range(4)) for a in range(4)]


def round_bits(q, bits=256):
    """q rounded to `bits` significant bits: a dyadic rational, so that the curvature fit's sum stays cheap; 256 bits is exact
    for every comparison made here."""
    if q == 0:
        return q
    e = bits - (abs(q.numerator).bit_length() - q.denominator.bit_length())
    return Fraction(round(q * 2 ** e), 2 ** e) if e >= 0 else Fraction(round(q / 2 ** -e) * 2 ** -e)


def exact_reference(xw, yw, n1, n2):
    """nav_msgs_path_frenet.py:44-86 from the samples xw, yw (0.5 m grid) in exact arithmetic: the two cubic fits, the curvature of
    the fitted cubics on the 0.25 m grid, its cubic fit.  Returns (K coefficients as Fractions, psi_start, e_y)."""
    xc = lsq_cubic(n1, 0.5, [Fraction(v) for v in xw]); yc = lsq_cubic(n1, 0.5, [Fraction(v) for v in yw])
    Km = []
    for g in range(n2):
        t = Fraction(g, 4)
        dx = xc[2] + 2 * xc[1] * t + 3 * xc[0] * t * t; dy = yc[2] + 2 * yc[1] * t + 3 * yc[0] * t * t
        ddx = 2 * xc[1] + 6 * xc[0] * t; ddy = 2 * yc[1] + 6 * yc[0] * t
        Km.append(round_bits((dx * ddy - dy * ddx) / (dx * dx + dy * dy)))
    K = lsq_cubic(n2, 0.25, Km)
    psi0 = math.atan2(yc[2], xc[2])      # the exact coefficients, rounded once by float()
    ey = -(-math.sin(psi0) * xw[0] + math.cos(psi0) * yw[0])
    return K, psi0, ey


# ---- 1. grid sizes and fit matrices
def test_fit_grid_sizes_match_numpy_arange():
    """The library sizes its fit grids as np.arange does: a window just above a multiple of the step has one more sample."""
    import emu_frenet as EF
    for w in WINDOWS:
        assert EF.fit_grid_sizes(w) == (np.arange(0.0, w, 0.5).size, np.arange(0.0, w, 0.25).size), w


def test_cubic_fit_matrix_is_exact():
    """cubic_fit_matrix (long-double normal equations on scaled columns) against (V'V)^-1 V' in exact rationals, for every grid
    size the windows above give, up to n = 2000."""
    import emu_frenet as EF
    sizes = sorted({(n, step) for w in WINDOWS for n, step in zip(EF.fit_grid_sizes(w), (0.5, 0.25))})
    assert (2000, 0.25) in sizes
    for n, step in sizes:
        Gi, V = exact_fit(n, step)
        P = EF.cubic_fit_matrix(n, step)
        for a in range(4):
            row = [sum(Gi[a][b] * V[g][b] for b in range(4)) for g in range(n)]
            d = max(abs(Fraction(P[a, g]) - row[g]) for g in range(n)) / max(abs(v) for v in row)
            observe("fit_matrix", float(d), FIT_MATRIX_BAR)


# ---- 2. one control period's reference
def reference_poses(tr, window):
    """On the path at index 0; mid-path 0.7 m and 3 m to either side with heading errors up to +-0.5 rad; near the end, so that
    the window straddles the last sample and np.interp clamps part of it."""
    j = tr.shape[0] // 2
    nrm = np.array([-np.sin(tr[j, 3]), np.cos(tr[j, 3])])
    poses = [tr[0, [4, 5, 3]]]
    for off, dpsi in ((0.7, 0.5), (-0.7, -0.3), (3.0, 0.2), (-3.0, -0.5)):
        xy = tr[j, 4:6] + off * nrm
        poses.append((xy[0], xy[1], tr[j, 3] + dpsi))
    je = int(np.searchsorted(tr[:, 6], tr[-1, 6] - 0.5 * min(window, 40.0)))
    poses.append(tr[je, [4, 5, 3]] + np.array([0.3, -0.2, 0.1]))
    return np.array(poses)


@pytest.mark.parametrize("window", [4.0, 40.0, 40.3, 500.0])
def test_frenet_reference_is_exact(oracle, tables, window):
    """frenet_reference on one emulated warp against the exact chain from the same samples.  The samples themselves are what
    numpy gives (np.argmin, np.interp, the rotation into the vehicle frame): bit for bit."""
    import emu as E
    import emu_frenet as EF
    kc = E.kcfg_from_oracle(oracle.default_cfg_frenet(8))
    n1, n2 = EF.fit_grid_sizes(window)
    grid = [Fraction(g, 4) for g in range(n2)]
    pe = lambda c, t: ((c[0] * t + c[1]) * t + c[2]) * t + c[3]
    for p, tr in enumerate(tables):
        poses = reference_poses(tr, window)
        r = EF.frenet_reference(kc, tr, poses, window, ey_from_path=True)
        r0 = EF.frenet_reference(kc, tr, poses, window, ey_from_path=False)
        assert np.array_equal(r0["kc"], r["kc"]) and np.array_equal(r0["psi0"], r["psi0"]) and (r0["ey"] == 0.0).all()
        assert tr[r["nearest"][-1], 6] + window > tr[-1, 6]      # the last pose's window reaches past the path end
        for m, (X, Y, yaw) in enumerate(poses):
            i = int(np.argmin((tr[:, 4] - X) ** 2 + (tr[:, 5] - Y) ** 2))
            assert r["nearest"][m] == i, (p, m)
            sq = tr[i, 6] + np.arange(0.0, window, 0.5)
            dx, dy = np.interp(sq, tr[:, 6], tr[:, 4]) - X, np.interp(sq, tr[:, 6], tr[:, 5]) - Y
            c, s = math.cos(yaw), math.sin(yaw)
            assert np.array_equal(r["xw"][m], c * dx + s * dy) and np.array_equal(r["yw"][m], -s * dx + c * dy), (p, m)
            K, psi0, ey = exact_reference(r["xw"][m], r["yw"][m], n1, n2)
            Ke = [pe(K, t) for t in grid]
            kk = [Fraction(v) for v in r["kc"][m]]
            dK = max(abs(pe(kk, t) - k) for t, k in zip(grid, Ke)) / max(abs(k) for k in Ke)
            observe("K_w%g" % window, float(dK), K_BAR[window])
            observe("psi_start", abs(r["psi0"][m] - psi0), PSI_BAR)
            observe("e_y", abs(r["ey"][m] - ey), EY_BAR)


# ---- 3. the closed loop, iterate for iterate
T = 6

# id: (N, window, ey_from_path, weights (oracle slot order) or None, fleet size; path_of cycles over the three paths when B = 7)
LOOP_CASES = {
    "N3":         (3, 40.0, True, None, 3),
    "N8":         (8, 40.0, True, None, 3),
    "N20":        (20, 40.0, True, None, 3),
    "N31":        (31, 40.0, True, None, 3),
    "N8_w4":      (8, 4.0, True, None, 3),
    "N8_w40.3":   (8, 40.3, True, None, 3),
    "N8_w500":    (8, 500.0, True, None, 3),
    "N8_ey0":     (8, 40.0, False, None, 3),
    "N8_weights": (8, 40.0, True, (0.0, 4.0, 25.0, 1.5, 40.0, 3000.0, 0.5, 2.0), 3),
    "N8_fleet7":  (8, 40.0, True, None, 7),
}


def loop_fleet(tables, B, seed):
    """B vehicles beside the path (0.3 m, 0.03 rad noise), spread along it; B = 7: paths 0, 1, 2, 0, ... and a last block of
    four vehicles that is partly full."""
    rng = np.random.default_rng(seed)
    path_of = (np.arange(B) % 3).astype(np.int32) if B == 7 else np.zeros(B, dtype=np.int32)
    idx = [300, 2500, 3900, 1200, 4700, 800, 3100]
    pose0 = np.array([tables[p][idx[v], [4, 5, 3]] + rng.normal(scale=[0.3, 0.3, 0.03]) for v, p in enumerate(path_of)])
    return pose0, path_of


def oracle_logs(oracle, tables, case, pose0, path_of, max_iter):
    N, window, ey_from_path, w, B = case
    cfg = oracle.default_cfg_frenet(N, weights=w, max_iter=max_iter)
    return np.stack([oracle.closed_loop_frenet(cfg, tables[path_of[v]], pose0[v], T, window, 8.0, ey_from_path) for v in range(B)], axis=1)


def compare_loops(name, glog, olog, capped):
    """glog, olog (T, B, 8).  Capped: equal statuses and iteration counts in every period, poses and commands to ITER_BAR; else
    equal statuses, |d iters| <= 1, commands to U_BAR."""
    assert np.array_equal(glog[:, :, 6], olog[:, :, 6]), (name, glog[:, :, 6], olog[:, :, 6])
    if capped:
        assert np.array_equal(glog[:, :, 7], olog[:, :, 7]), (name, glog[:, :, 7], olog[:, :, 7])
        assert (olog[:, :, 6] == 3).mean() >= 0.9, name
        observe(name, (np.abs(glog[:, :, 0:6] - olog[:, :, 0:6]) / np.maximum(1.0, np.abs(olog[:, :, 0:6]))).max(), ITER_BAR)
    else:
        assert (olog[:, :, 6] == 0).mean() >= 0.9, name
        assert np.abs(glog[:, :, 7] - olog[:, :, 7]).max() <= 1, (name, glog[:, :, 7], olog[:, :, 7])
        observe(name, np.abs(glog[:, :, 4:6] - olog[:, :, 4:6]).max(), U_BAR)


@pytest.mark.parametrize("form", ["fused", "pipeline"])
@pytest.mark.parametrize("case", list(LOOP_CASES))
def test_closed_loop_matches_oracle(oracle, tables, case, form):
    """rollout_group_frenet (fused) and the per-period pipeline against oracle.closed_loop_frenet, vehicle by vehicle, at
    max_iter = 1, 3 and the default cap.  The fleet runs three distinct path tables (vehicle -> table through path_of)."""
    import emu as E
    import emu_frenet as EF
    c = LOOP_CASES[case]
    N, window, ey_from_path, w, B = c
    pose0, path_of = loop_fleet(tables, B, seed=N)
    for max_iter in (1, 3, None):
        cfg = oracle.default_cfg_frenet(N, weights=w, max_iter=max_iter)
        glog, _ = EF.rollout_frenet3(E.kcfg_from_oracle(cfg), tables, pose0, path_of, T, window=window, target_vel=8.0,
                                     ey_from_path=ey_from_path, tpp=form == "pipeline")
        olog = oracle_logs(oracle, tables, c, pose0, path_of, max_iter)
        compare_loops("loop_%s" % ("capped" if max_iter else "full"), glog, olog, max_iter is not None)
