"""CPU check of per-vehicle cost weights in the Frenet closed loop (mpcb200_rollout_frenet_w): the PW = 1 forms of the kernel sources
on the warp emulator (tests/emu/emu_frenet_weights.py), under its shared-memory race check -- the fused loop
(rollout_group_frenet<MET, 1>) and the per-period pipeline (TppSolverT<1, 1> warm-started in place).

  * against oracle.closed_loop_frenet with each vehicle's own row, iterate for iterate at max_iter = 1 and 3, then uncapped (the
    scheme and bars of test_frenet_closed_loop_emu.py);
  * every row equal to the handle's weights: the PW = 0 loop's log bit for bit;
  * a fleet mixing four rows: each vehicle as the PW = 0 loop with its row as the handle's weights, bit for bit;
  * MET = 1 with rows: the log of MET = 0, and metrics equal to closed_loop.tracking_metrics of that log, bit for bit."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

from test_frenet_closed_loop_emu import compare_loops, loop_fleet   # noqa: E402

T = 6
W_DEFAULT = np.array([9.0, 10.0, 0.5, 100.0, 1000.0, 0.0, 0.0])   # MKZMPCPathFollowerFrenet.jl:51-58, set_cost_frenet's order


def weight_rows(B, seed):
    """B rows: the five non-zero defaults times 10^U(-1, 1); ca and cd (0 by default) log-uniform in [0.1, 10]; row 0 keeps
    ca = cd = 0."""
    rng = np.random.default_rng(seed)
    base = np.where(W_DEFAULT > 0, W_DEFAULT, 1.0)
    rows = base * 10.0 ** rng.uniform(-1.0, 1.0, size=(B, 7))
    rows[0, 5:] = 0.0
    return rows


@pytest.fixture(scope="module")
def tables():
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    return [GPSRefTrajectory(mat_filename=p).trajectory for p in (1, 2, 3)]


@pytest.fixture(autouse=True)
def _race_check():
    import emu_frenet_weights as EFW
    EFW.race_check(True)
    yield
    assert EFW.race_count() == 0


def kcfg(oracle, N, row=None, max_iter=None):
    import emu as E
    return E.kcfg_from_oracle(oracle.default_cfg_frenet(N, weights=None if row is None else (0.0,) + tuple(row), max_iter=max_iter))


# id: (N, fleet size; B = 7 cycles over the three paths)
CASES = {"N3": (3, 3), "N8": (8, 3), "N20": (20, 3), "N8_fleet7": (8, 7)}


@pytest.mark.parametrize("form", ["fused", "pipeline"])
@pytest.mark.parametrize("case", list(CASES))
def test_weighted_loop_matches_oracle(oracle, tables, case, form):
    """Each vehicle with its own row against oracle.closed_loop_frenet with that row, at max_iter = 1, 3 and the default cap."""
    import emu_frenet_weights as EFW
    N, B = CASES[case]
    pose0, path_of = loop_fleet(tables, B, seed=N)
    rows = weight_rows(B, seed=N)
    for max_iter in (1, 3, None):
        glog, _ = EFW.rollout_frenet_w(kcfg(oracle, N, max_iter=max_iter), tables, pose0, path_of, T, rows, tpp=form == "pipeline")
        olog = np.stack([oracle.closed_loop_frenet(oracle.default_cfg_frenet(N, weights=(0.0,) + tuple(rows[v]), max_iter=max_iter),
                                                   tables[path_of[v]], pose0[v], T, 40.0, 8.0, True) for v in range(B)], axis=1)
        compare_loops("loop_%s" % ("capped" if max_iter else "full"), glog, olog, max_iter is not None)


@pytest.mark.parametrize("form", ["fused", "pipeline"])
def test_equal_rows_reproduce_unweighted_loop(oracle, tables, form):
    """Rows equal to the handle's weights: the PW = 0 loop's log and final state, bit for bit."""
    import emu_frenet as EF
    import emu_frenet_weights as EFW
    k = kcfg(oracle, 8)
    pose0, path_of = loop_fleet(tables, 7, seed=8)
    log, final = EFW.rollout_frenet_w(k, tables, pose0, path_of, T, np.tile(W_DEFAULT, (7, 1)), tpp=form == "pipeline")
    plog, pfinal = EF.rollout_frenet3(k, tables, pose0, path_of, T, tpp=form == "pipeline")
    assert np.array_equal(log, plog) and np.array_equal(final, pfinal)


@pytest.mark.parametrize("form", ["fused", "pipeline"])
def test_mixed_rows_equal_single_row_fleets(oracle, tables, form):
    """A fleet of eight vehicles over four rows: every vehicle as in the PW = 0 loop whose handle weights are its row."""
    import emu_frenet as EF
    import emu_frenet_weights as EFW
    rows4 = weight_rows(4, seed=3)
    rng = np.random.default_rng(5)
    path_of = np.zeros(8, dtype=np.int32)
    pose0 = np.array([tables[0][i, [4, 5, 3]] for i in (300, 900, 1500, 2100, 2700, 3300, 3900, 4500)]) + rng.normal(
        scale=[0.3, 0.3, 0.03], size=(8, 3))
    which = np.arange(8) % 4
    log, final = EFW.rollout_frenet_w(kcfg(oracle, 8), tables, pose0, path_of, T, rows4[which], tpp=form == "pipeline")
    for r in range(4):
        sel = which == r
        plog, pfinal = EF.rollout_frenet3(kcfg(oracle, 8, row=rows4[r]), tables, pose0[sel], path_of[sel], T, tpp=form == "pipeline")
        assert np.array_equal(log[:, sel], plog) and np.array_equal(final[sel], pfinal), r


def test_metrics_with_rows_match_log(oracle, tables):
    """rollout_group_frenet<1, 1>: the log of rollout_group_frenet<0, 1>, and metrics equal to tracking_metrics of it."""
    import emu_frenet_weights as EFW
    from mkz_mpc_path_follower_b200.closed_loop import tracking_metrics
    pose0, _ = loop_fleet(tables, 3, seed=8)
    pose0 = np.vstack([pose0, pose0 + [0.4, -0.3, 0.05]])
    path_of = np.zeros(6, dtype=np.int32)
    rows = weight_rows(6, seed=11)
    k = kcfg(oracle, 8)
    log, final, met = EFW.rollout_frenet_w(k, tables, pose0, path_of, T, rows, metrics=True)
    plog, pfinal = EFW.rollout_frenet_w(k, tables, pose0, path_of, T, rows)
    assert np.array_equal(log, plog) and np.array_equal(final, pfinal)
    assert np.array_equal(met, tracking_metrics(log, tables[0]), equal_nan=True)
    assert (met[:, 0] == T).all() and (met[:, 11] == -1).all()
