"""The Frenet closed loop on the GPU (mpcb200_rollout_frenet) against oracle.closed_loop_frenet, iterate for iterate.

The oracle's loop shares nothing with the library: its plant is the oracle's, its fits are np.polyfit, its solves are the
oracle's interior-point code.  Every row runs the C ABI at max_iter = 3 (each period's solve stops at an interior iterate, so a
wrong curvature fit, e_y or Newton step shows in the published command), then at the handle's default cap.  Capped: equal
statuses and iteration counts in every period, most periods capped, poses and commands within the row's bar relative to
max(1, |x|).  Uncapped: equal statuses, iteration counts within one, commands within U_BAR.

Which instantiation each row reaches (csrc/mpc_b200.cu: rollout_enqueue):

  fused_N3, fused_N8, fused_N20, fused_N31      mpc_rollout_frenet_kernel (rollout_group_frenet), window 40 m
  pipeline_N8, pipeline_N31                     rollout_frenet_ref_kernel + rollout_solve_tpp_kernel<1, 0>, set_large_batch_path(1)
  fused_N8_w4, fused_N8_w40.3, fused_N8_w500    mpc_rollout_frenet_kernel, other fit windows (other fit matrices and grid sizes)
  fused_N8_ey0                                  ey_from_path = 0 (the reference node's e_y)
  fused_N8_cost                                 weights set by set_cost_frenet
  fleet7                                        B = 7 vehicles over three set_path tables: vehicle -> table through path_of,
                                                and a last block of four warps that is partly full

Bars: the GPU build contracts multiply-adds and uses its own sincos, atan2 and reciprocal, so it does not round like the host build
of the emulator (test_frenet_closed_loop_emu.py).  The largest relative difference per row over all periods and
vehicles, measured on a B200 at a 1,000 W power limit, is in BARS' comments; each bar is 10x that, rounded up to one digit.
`pytest -s` prints the observed table; a new row has no bar until its floor is measured.  Measured floors: 1e-16 to 4e-15.
Sensitivity: with `3.0 * xc[0]` made `2.0 * xc[0]` or the curvature grid 0.25 m made 0.5 m in frenet_reference, the rows differ by
1e-8 to 2e-2 (or their iteration counts differ); with e_y computed from the wrong lane, every row but fused_N8_ey0 differs by 6e-5
or more; with e_y negated in rollout_solve_tpp_kernel<1>, both pipeline rows differ by 0.2 or more."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

T = 6
U_BAR = 1e-8     # uncapped: |du|

# id: (instantiation, N, window, ey_from_path, set_cost_frenet weights or None, fleet size, per-period pipeline)
ROWS = {
    "fused_N3":       ("mpc_rollout_frenet_kernel", 3, 40.0, True, None, 3, False),
    "fused_N8":       ("mpc_rollout_frenet_kernel", 8, 40.0, True, None, 3, False),
    "fused_N20":      ("mpc_rollout_frenet_kernel", 20, 40.0, True, None, 3, False),
    "fused_N31":      ("mpc_rollout_frenet_kernel", 31, 40.0, True, None, 3, False),
    "pipeline_N8":    ("rollout_solve_tpp_kernel<1, 0>", 8, 40.0, True, None, 3, True),
    "pipeline_N31":   ("rollout_solve_tpp_kernel<1, 0>", 31, 40.0, True, None, 3, True),
    "fused_N8_w4":    ("mpc_rollout_frenet_kernel", 8, 4.0, True, None, 3, False),
    "fused_N8_w40.3": ("mpc_rollout_frenet_kernel", 8, 40.3, True, None, 3, False),
    "fused_N8_w500":  ("mpc_rollout_frenet_kernel", 8, 500.0, True, None, 3, False),
    "fused_N8_ey0":   ("mpc_rollout_frenet_kernel", 8, 40.0, False, None, 3, False),
    "fused_N8_cost":  ("mpc_rollout_frenet_kernel", 8, 40.0, True, (4.0, 25.0, 1.5, 40.0, 3000.0, 0.5, 2.0), 3, False),
    "fleet7":         ("mpc_rollout_frenet_kernel", 8, 40.0, True, None, 7, False),
}

# row id -> bar: 10x the largest relative difference observed on a B200 (1,000 W), rounded up to one digit
BARS = {
    "fleet7":          6e-15,    # observed 5.97e-16
    "fused_N20":       3e-14,    # observed 2.37e-15
    "fused_N3":        4e-15,    # observed 3.33e-16
    "fused_N31":       4e-14,    # observed 3.72e-15
    "fused_N8":        4e-15,    # observed 3.33e-16
    "fused_N8_cost":   2e-14,    # observed 1.30e-15
    "fused_N8_ey0":    1e-15,    # observed 9.71e-17
    "fused_N8_w4":     8e-15,    # observed 7.22e-16
    "fused_N8_w40.3":  6e-15,    # observed 5.00e-16
    "fused_N8_w500":   2e-14,    # observed 1.14e-15
    "pipeline_N31":    4e-14,    # observed 3.71e-15
    "pipeline_N8":     3e-15,    # observed 2.78e-16
}

OBSERVED = {}        # row id -> largest relative difference seen (printed at the end of the module)


def bar(row):
    return BARS[row]       # a new row needs its floor measured first


def observe(row, d):
    OBSERVED[row] = max(OBSERVED.get(row, 0.0), float(d)) if d == d else float("nan")
    assert d <= bar(row), (row, d, bar(row))


@pytest.fixture(scope="module", autouse=True)
def _print_observed():
    yield
    for row in sorted(OBSERVED):
        print("observed %-16s %.2e  (bar %.0e)" % (row, OBSERVED[row], bar(row)))


@pytest.fixture(scope="module")
def capi():
    from mkz_mpc_path_follower_b200 import capi as c
    c.lib()
    return c


@pytest.fixture(scope="module")
def tables():
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    return [GPSRefTrajectory(mat_filename=p).trajectory for p in (1, 2, 3)]


def gpu_rollout(capi, tables, row, pose0, path_of, max_iter):
    _, N, window, ey_from_path, w, B, pipeline = ROWS[row]
    s = capi.FrenetSolver(N) if max_iter is None else capi.FrenetSolver(N, max_iter=max_iter)
    try:
        cap = s.cfg.max_iter
        s.set_large_batch_path(1 if pipeline else 0)
        if w is not None:
            s.set_cost(np.array(w))
        for i, tr in enumerate(tables):
            s.set_path(i, tr)
        out = s.rollout(pose0, path_of, T, window=window, target_vel=8.0, ey_from_path=ey_from_path)
        assert s.stats()["kernel_launches"] == (3 * T + 1 if pipeline else 1)
    finally:
        s.close()
    return out["log"], cap


@pytest.mark.parametrize("row", list(ROWS))
def test_frenet_rollout_iterates(capi, oracle, tables, row):
    from test_frenet_closed_loop_emu import loop_fleet
    _, N, window, ey_from_path, w, B, pipeline = ROWS[row]
    pose0, path_of = loop_fleet(tables, B, seed=N)
    ow = None if w is None else (0.0,) + tuple(w)          # the oracle's slot order: (0, cey, cep, cev, cda, cdd, ca, cd)
    for max_iter in (3, None):
        glog, cap = gpu_rollout(capi, tables, row, pose0, path_of, max_iter)
        cfg = oracle.default_cfg_frenet(N, weights=ow, max_iter=cap)
        olog = np.stack([oracle.closed_loop_frenet(cfg, tables[path_of[v]], pose0[v], T, window, 8.0, ey_from_path)
                         for v in range(B)], axis=1)
        assert np.array_equal(glog[:, :, 6], olog[:, :, 6]), (row, glog[:, :, 6], olog[:, :, 6])
        if max_iter is not None:
            assert np.array_equal(glog[:, :, 7], olog[:, :, 7]), (row, glog[:, :, 7], olog[:, :, 7])
            assert (olog[:, :, 6] == 3).mean() >= 0.9, row
            observe(row, (np.abs(glog[:, :, 0:6] - olog[:, :, 0:6]) / np.maximum(1.0, np.abs(olog[:, :, 0:6]))).max())
        else:
            assert (olog[:, :, 6] == 0).mean() >= 0.9, row
            assert np.abs(glog[:, :, 7] - olog[:, :, 7]).max() <= 1, (row, glog[:, :, 7], olog[:, :, 7])
            assert np.abs(glog[:, :, 4:6] - olog[:, :, 4:6]).max() <= U_BAR, row
