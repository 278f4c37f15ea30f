"""mpcb200_solve_batch_frenet_on_path on the kernel sources (compiled for the host, tests/emu) against references that share nothing
with them.

The call is the reference pass on_path_frenet_ref_kernel (frenet_on_path_problem: frenet_reference from the pose, K(s) and
(0, e_y, -psi_start, v) into two [B][4] rows), then the solve kernels of mpcb200_solve_batch_frenet on those rows.  Here:

  * the reference pass against frenet_on_path_ref.frenet_on_path (np.argmin, np.interp, oracle.frenet_fit: the reference step of
    oracle.closed_loop_frenet), over three path tables in one batch, windows 4, 40, 40.3 and 500 m, poses on, beside and across
    the path, near its end and kilometres away, with e_y from the path and e_y = 0;
  * the emulated warp solver (N = 3, 8, 20, 31; N = 40 on a two-warp team) and the thread-per-problem solver source, run on the
    pass's own rows, against oracle.solve_batch_frenet on the reference's rows, iterate for iterate at max_iter 1 and 3 and
    uncapped, with and without per-problem weight rows;
  * a path id that was never set: NaN rows, the solve of those rows ends, and the neighbours are unaffected;
  * frenet_on_path_ref itself: a loop built on it reproduces oracle.closed_loop_frenet bit for bit.

Bars are 10x the largest difference measured with the host build (g++ -O1, no contraction), rounded up to one digit.  Measured,
near the path / 2 km away:
  K(s) on the 0.25 m grid, relative to max |K|: w = 4: 6.7e-12 / 1.6e-9; 40: 1.2e-12 / 4.6e-11; 40.3: 1.1e-12 / 1.2e-11;
      500: 2.2e-10 (the pose near the end: most samples are the last point, max |K| is small) / 2.7e-14
  psi_start, absolute: 4.1e-15 / 1.7e-12;  e_y relative to max(1, |e_y|): 6.5e-16 / 1.6e-12
  solves: capped iterates 5.3e-14 relative to max(1, |x|), uncapped commands 2.4e-16; their bar is that of the iterate tests, 1e-10.
`pytest -s` prints the largest difference seen per check next to its bar."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

from frenet_on_path_ref import batch3, far_poses, frenet_on_path, frenet_on_path_batch  # noqa: E402

# bars per window for poses near the path (on, beside, across, near the end) and for the poses 2 km away, whose window in the
# vehicle frame lies ~2 km off the origin of the fit (the cubic fits then cancel ~2,000 m constants)
K_BAR = {"near": {4.0: 7e-11, 40.0: 2e-11, 40.3: 2e-11, 500.0: 3e-9}, "far": {4.0: 2e-8, 40.0: 5e-10, 40.3: 2e-10, 500.0: 3e-13}}
PSI_BAR = {"near": 5e-14, "far": 2e-11}
EY_BAR = {"near": 7e-15, "far": 2e-11}
ITER_BAR = 1e-10
U_BAR = 1e-10

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


def compare_reference(name, tables, pose, path_of, window, k, st, K, S):
    grid = np.arange(0.0, window, 0.25)
    far = far_poses(tables, pose, path_of)
    for b in range(pose.shape[0]):
        c = "far" if far[b] else "near"
        Ke = np.polyval(K[b], grid)
        observe("K_w%g_%s" % (window, c), np.abs(np.polyval(k[b], grid) - Ke).max() / np.abs(Ke).max(), K_BAR[c][window])
        observe("psi_start_" + c, abs(st[b, 2] - S[b, 2]), PSI_BAR[c])
        observe("e_y_" + c, abs(st[b, 1] - S[b, 1]) / max(1.0, abs(S[b, 1])), EY_BAR[c])
        assert st[b, 0] == 0.0 and st[b, 3] == pose[b, 3], (name, b)


# ---- 1. the reference pass
@pytest.mark.parametrize("window", [4.0, 40.0, 40.3, 500.0])
def test_reference_pass_matches_oracle(oracle, tables, window):
    """frenet_on_path_problem on one emulated warp per problem against the reference step of oracle.closed_loop_frenet, three
    tables in one batch, e_y from the path and e_y = 0 (which changes nothing else, bit for bit)."""
    import emu as E
    import emu_frenet_on_path as EP
    kc = E.kcfg_from_oracle(oracle.default_cfg_frenet(8))
    pose, path_of = batch3(tables, window)
    k1, s1 = EP.frenet_on_path(kc, tables, pose, path_of, window, ey_from_path=True)
    k0, s0 = EP.frenet_on_path(kc, tables, pose, path_of, window, ey_from_path=False)
    assert np.array_equal(k0, k1) and np.array_equal(s0[:, [0, 2, 3]], s1[:, [0, 2, 3]]) and (s0[:, 1] == 0.0).all()
    K, S = frenet_on_path_batch(oracle, tables, pose, path_of, window, True)
    compare_reference("ey1", tables, pose, path_of, window, k1, s1, K, S)
    assert far_poses(tables, pose, path_of).sum() == 3      # the kilometre-away poses are in the batch


# ---- 2. the solves of the pass's rows, iterate for iterate
# id: (N, window, weight rows or None, thread-per-problem source)
SOLVE_CASES = {
    "N3": (3, 40.0, False, False),
    "N8": (8, 40.0, False, False),
    "N20": (20, 40.0, False, False),
    "N31": (31, 40.0, False, False),
    "N40_team2": (40, 40.0, False, False),
    "N8_w500": (8, 500.0, False, False),
    "N8_weights": (8, 40.0, True, False),
    "N8_tpp": (8, 40.0, False, True),
    "N20_tpp_weights": (20, 40.0, True, True),
}


def solve_batch(E, EW, kc, st, k, v_des, u_prev, w, tpp):
    if w is None:
        return E.solve_batch_frenet(kc, st, k, v_des, u_prev, want_traj=True, tpp=tpp)
    return EW.solve_batch_frenet_w(kc, st, k, v_des, u_prev, w, want_traj=True, tpp=tpp)


def oracle_solves(oracle, N, max_iter, S, K, v_des, u_prev, w):
    """oracle.solve_batch_frenet problem by problem with each problem's own row (the oracle's XY slot order: 0 on s first)."""
    out = {f: [] for f in ("u0", "cost", "status", "iters", "traj")}
    for b in range(S.shape[0]):
        cfg = oracle.default_cfg_frenet(N, weights=None if w is None else (0.0,) + tuple(w[b]), max_iter=max_iter)
        o = oracle.solve_batch_frenet(cfg, S[b:b + 1], K[b:b + 1], v_des[b:b + 1], u_prev[b:b + 1], want_traj=True)
        for f in out:
            out[f].append(o[f][0])
    return {f: np.array(v) for f, v in out.items()}


@pytest.mark.parametrize("case", list(SOLVE_CASES))
def test_solves_of_the_pass_match_oracle(oracle, tables, case):
    """The warp solver (team of team_warps(N) warps) or the thread-per-problem solver on the emulated pass's rows against the oracle
    on the reference step's rows, at max_iter 1 and 3 (every problem stops at an interior iterate) and uncapped."""
    import emu as E
    import emu_frenet_on_path as EP
    import emu_weights as EW
    N, window, weighted, tpp = SOLVE_CASES[case]
    rng = np.random.default_rng(N)
    idx = [400, 1900, 3300]
    pose = np.array([(*tables[p][idx[p], [4, 5, 3]], 0.0) for p in (0, 1, 2, 0, 1, 2)])
    pose[:, :3] += rng.normal(scale=[0.4, 0.4, 0.05], size=(6, 3))
    pose[:, 3] = rng.uniform(2.0, 9.0, 6)
    path_of = np.array([0, 1, 2, 0, 1, 2], dtype=np.int32)
    u_prev = rng.uniform(-0.05, 0.05, (6, 2))
    v_des = rng.uniform(6.0, 10.0, 6)
    w = rng.uniform(0.5, 2.0, (6, 7)) * np.array([9.0, 10.0, 0.5, 100.0, 1000.0, 0.5, 0.5]) if weighted else None
    K, S = frenet_on_path_batch(oracle, tables, pose, path_of, window, True)
    for max_iter in (1, 3, None):
        cfg = oracle.default_cfg_frenet(N, max_iter=max_iter)
        kc = E.kcfg_from_oracle(cfg)
        k, st = EP.frenet_on_path(kc, tables, pose, path_of, window)
        g = solve_batch(E, EW, kc, st, k, v_des, u_prev, w, tpp)
        o = oracle_solves(oracle, N, max_iter, S, K, v_des, u_prev, w)
        assert np.array_equal(g["status"], o["status"]), (case, max_iter, g["status"], o["status"])
        assert np.array_equal(g["iters"], o["iters"]), (case, max_iter, g["iters"], o["iters"])
        if max_iter is not None:
            assert (o["status"] == 3).all(), (case, max_iter)
            observe("iterate_capped", (np.abs(g["traj"] - o["traj"]) / np.maximum(1.0, np.abs(o["traj"]))).max(), ITER_BAR)
        else:
            assert (o["status"] == 0).all(), (case, o["status"])
            observe("u0_uncapped", np.abs(g["u0"] - o["u0"]).max(), U_BAR)


# ---- 3. a path id that was never set
@pytest.mark.parametrize("tpp", [False, True], ids=["warp", "tpp"])
def test_unset_path_id(oracle, tables, tpp):
    """Problems on a table that was never set and on ids outside 0..2 get NaN rows; the solve of those rows ends (within the cap)
    and the other problems' rows and answers are those of the same batch without them, bit for bit."""
    import emu as E
    import emu_frenet_on_path as EP
    kc = E.kcfg_from_oracle(oracle.default_cfg_frenet(8))
    pose = np.array([(*tables[0][500, [4, 5, 3]], 5.0), (*tables[1][800, [4, 5, 3]], 5.0), (*tables[0][900, [4, 5, 3]], 6.0),
                     (*tables[0][1200, [4, 5, 3]], 7.0), (*tables[0][1500, [4, 5, 3]], 7.0)])
    path_of = np.array([0, 2, 0, -1, 3], dtype=np.int32)
    k, st = EP.frenet_on_path(kc, tables, pose, path_of, 40.0, unset=(2,))
    bad = np.array([False, True, False, True, True])
    assert np.isnan(k[bad]).all() and np.isnan(st[bad]).all() and np.isfinite(k[~bad]).all() and np.isfinite(st[~bad]).all()
    k2, st2 = EP.frenet_on_path(kc, tables, pose[~bad], path_of[~bad], 40.0, unset=(2,))
    assert np.array_equal(k[~bad], k2) and np.array_equal(st[~bad], st2)
    u_prev = np.zeros((5, 2)); v_des = np.full(5, 8.0)
    g = E.solve_batch_frenet(kc, st, k, v_des, u_prev, tpp=tpp)
    g2 = E.solve_batch_frenet(kc, st2, k2, v_des[~bad], u_prev[~bad], tpp=tpp)
    for f in ("u0", "cost", "status", "iters"):
        assert np.array_equal(g[f][~bad], g2[f]), f
    assert (g["iters"][bad] <= kc.max_iter).all()


# ---- 4. the reference itself
def test_reference_reproduces_oracle_closed_loop(oracle, tables):
    """A closed loop on frenet_on_path_ref (oracle.plant_step, solve_batch_frenet from the previous solution) gives the log of
    oracle.closed_loop_frenet bit for bit: the reference step is the one the oracle's loop takes."""
    N, T, window = 8, 5, 40.0
    cfg = oracle.default_cfg_frenet(N)
    for p, tr in enumerate(tables):
        pose0 = tr[700 + 900 * p, [4, 5, 3]] + np.array([0.3, -0.2, 0.05])
        st = np.array([pose0[0], pose0[1], pose0[2], 0.0, 0.0, 0.0, 0.0, 0.0])
        acc = df = 0.0
        u_prev = np.zeros((1, 2)); warm = np.zeros((1, 6 * N + 4)); log = np.zeros((T, 8))
        for t in range(T):
            for _ in range(10):
                st = oracle.plant_step(st, acc, df)
            K, S = frenet_on_path(oracle, tr, st[:4], window, True)
            o = oracle.solve_batch_frenet(cfg, S[None], K[None], np.array([8.0]), u_prev, warm=warm)
            acc, df = float(o["u0"][0, 0]), float(o["u0"][0, 1])
            u_prev[0] = (df, acc)
            log[t] = (st[0], st[1], st[2], st[3], acc, df, o["status"][0], o["iters"][0])
        assert np.array_equal(log, oracle.closed_loop_frenet(cfg, tr, pose0, T, window, 8.0, True)), p
