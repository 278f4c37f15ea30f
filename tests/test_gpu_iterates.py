"""Every solve and rollout kernel the library can launch, checked iterate for iterate against the oracle through the C ABI.

The endpoint checks of the other GPU tests (same status, |du| <= 1e-5) cannot see a wrong Newton step: the filter line search
still ends at the same KKT point.  Here each kernel returns its trajectory after max_iter = k iterations, k = 1, 2, 3, 5, 10
(status UserLimit), and that iterate must be the oracle's to the row's bar, relative to max(1, |traj|).  Then a full solve:
equal statuses, equal iteration counts wherever the oracle needs at most 60 iterations, the same command where Optimal.

Which instantiation each row reaches (csrc/mpc_b200.cu: team_kernel, rollout_kernel, launch_solve, rollout_enqueue):

  solve rows (SOLVE_ROWS)                                     rollout rows (ROLLOUT_ROWS), max_iter = 3 in every period
  mpc_solve_kernel<0|1>            XY, N = 3, 8, 20, 31       mpc_rollout_kernel<0|1>           N = 8, fleets below the switch
  mpc_solve_long_kernel<2, 0, 0|1> XY, N = 32, 63             mpc_rollout_long_kernel<2, 0|1>   N = 40
  mpc_solve_long_kernel<3, 0, 0|1> XY, N = 64, 95             mpc_rollout_long_kernel<3, 0|1>   N = 80
  mpc_solve_frenet_kernel<3|4, 0|1> Frenet, N = 8, 20, both   rollout_solve_tpp_kernel<0, 0|1>  N = 8, set_large_batch_path(1)
                                   block sizes forced by MPCB200_FRENET_WPB
  mpc_solve_long_kernel<2, 1, 0|1> Frenet, N = 32, 63
  mpc_solve_long_kernel<3, 1, 0|1> Frenet, N = 64, 95
  mpc_solve_tpp_kernel<0|1, 0|1>   both models, N = 8, 20, 40, set_large_batch_path(1) and B = 96 (host batches of at most 64
                                   problems always take the packed small-batch path, which launches the team kernels)
The team rows run B <= 64 host batches (the packed small-batch path and its CUDA graph); test_records_and_device_pointers runs
the same kernels through the unpacked path, with mpcb200_solve_batch_records and with device pointers.  Not covered here:
mpc_rollout_frenet_kernel and the Frenet per-period pipeline (rollout_frenet_ref_kernel, rollout_solve_tpp_kernel<1, 0>), which
test_gpu_frenet_closed_loop.py checks iterate for iterate against oracle.closed_loop_frenet, and the reference generators of the
on-path entry points, which launch the solve kernels above and are checked bit for bit against the host generator elsewhere.

Bars: the GPU build contracts multiply-adds and uses its own sincos and reciprocal, so it does not round like the host build of
the emulator (floor 1e-12).  The largest relative difference per row over k = 1, 2, 3, 5, 10 (k = 2, 5 for the constant sets;
every period for the rollouts), measured on a B200 at a 1,000 W power limit, is in BARS' comments; each bar is 10x that,
rounded up to one digit.  Every kernel is deterministic for a given build and batch.  `pytest -s` prints the observed table;
a new row has no bar until its floor is measured.  Measured floors: 1e-14 to 3e-11 for every row but one.  The outlier is
xy_tpp_N20_w (the weighted thread-per-problem XY kernel, mpc_solve_tpp_kernel<0, 1>) at 1.2e-10, four times the next row and
fifteen times its unweighted sibling at N = 8.  It matches what was seen when that kernel was added: the PW = 1 thread layout
is the one build whose results differ, at equal weights, from the unweighted build beyond the last bits.  Its bar is 10x its
own floor like every other row (2e-9), not widened to hide it; the source of the extra rounding has not been traced.
"""
import os

import numpy as np
import pytest

from test_iterates_emu import CONSTANT_SETS, FULL_ITERS, KS, Case, iterate_error, weight_rows

pytestmark = pytest.mark.gpu

U_BAR = 1e-8     # full solves: |du| where Optimal

# id: (instantiation, model, N, B, layout, weighted, warm start from the reference waypoints, Frenet warps per block)
SOLVE_ROWS = {
    "xy_N3":         ("mpc_solve_kernel<0>", 0, 3, 24, "team", False, False, None),
    "xy_N8_w":       ("mpc_solve_kernel<1>", 0, 8, 24, "team", True, False, None),
    "xy_N20":        ("mpc_solve_kernel<0>", 0, 20, 16, "team", False, False, None),
    "xy_N31_w":      ("mpc_solve_kernel<1>", 0, 31, 8, "team", True, False, None),
    "xy_N32":        ("mpc_solve_long_kernel<2, 0, 0>", 0, 32, 6, "team", False, True, None),
    "xy_N63_w":      ("mpc_solve_long_kernel<2, 0, 1>", 0, 63, 6, "team", True, True, None),
    "xy_N64_w":      ("mpc_solve_long_kernel<3, 0, 1>", 0, 64, 6, "team", True, True, None),
    "xy_N95":        ("mpc_solve_long_kernel<3, 0, 0>", 0, 95, 6, "team", False, True, None),
    "fr_N8_wpb3":    ("mpc_solve_frenet_kernel<3, 0>", 1, 8, 16, "team", False, False, 3),
    "fr_N8_wpb3_w":  ("mpc_solve_frenet_kernel<3, 1>", 1, 8, 16, "team", True, False, 3),
    "fr_N8_wpb4":    ("mpc_solve_frenet_kernel<4, 0>", 1, 8, 16, "team", False, False, 4),
    "fr_N8_wpb4_w":  ("mpc_solve_frenet_kernel<4, 1>", 1, 8, 16, "team", True, False, 4),
    "fr_N20_wpb3":   ("mpc_solve_frenet_kernel<3, 0>", 1, 20, 12, "team", False, False, 3),
    "fr_N20_wpb3_w": ("mpc_solve_frenet_kernel<3, 1>", 1, 20, 12, "team", True, False, 3),
    "fr_N20_wpb4":   ("mpc_solve_frenet_kernel<4, 0>", 1, 20, 12, "team", False, False, 4),
    "fr_N20_wpb4_w": ("mpc_solve_frenet_kernel<4, 1>", 1, 20, 12, "team", True, False, 4),
    "fr_N32_w":      ("mpc_solve_long_kernel<2, 1, 1>", 1, 32, 6, "team", True, False, None),
    "fr_N63":        ("mpc_solve_long_kernel<2, 1, 0>", 1, 63, 6, "team", False, False, None),
    "fr_N64":        ("mpc_solve_long_kernel<3, 1, 0>", 1, 64, 6, "team", False, False, None),
    "fr_N95_w":      ("mpc_solve_long_kernel<3, 1, 1>", 1, 95, 6, "team", True, False, None),
    "xy_tpp_N8":     ("mpc_solve_tpp_kernel<0, 0>", 0, 8, 96, "tpp", False, False, None),
    "xy_tpp_N20_w":  ("mpc_solve_tpp_kernel<0, 1>", 0, 20, 96, "tpp", True, False, None),
    "xy_tpp_N40":    ("mpc_solve_tpp_kernel<0, 0>", 0, 40, 96, "tpp", False, True, None),
    "fr_tpp_N8_w":   ("mpc_solve_tpp_kernel<1, 1>", 1, 8, 96, "tpp", True, False, None),
    "fr_tpp_N20":    ("mpc_solve_tpp_kernel<1, 0>", 1, 20, 96, "tpp", False, False, None),
    "fr_tpp_N40_w":  ("mpc_solve_tpp_kernel<1, 1>", 1, 40, 96, "tpp", True, False, None),
}

# id: (instantiation, N, weighted, per-period pipeline)
ROLLOUT_ROWS = {
    "fused_N8":      ("mpc_rollout_kernel<0>", 8, False, False),
    "fused_N8_w":    ("mpc_rollout_kernel<1>", 8, True, False),
    "long_N40":      ("mpc_rollout_long_kernel<2, 0>", 40, False, False),
    "long_N40_w":    ("mpc_rollout_long_kernel<2, 1>", 40, True, False),
    "long_N80":      ("mpc_rollout_long_kernel<3, 0>", 80, False, False),
    "long_N80_w":    ("mpc_rollout_long_kernel<3, 1>", 80, True, False),
    "pipeline_N8":   ("rollout_solve_tpp_kernel<0, 0>", 8, False, True),
    "pipeline_N8_w": ("rollout_solve_tpp_kernel<0, 1>", 8, True, True),
}

# row id -> bar: 10x the largest relative difference observed on a B200 (1,000 W), rounded up to one digit
BARS = {
    "fr_N20_wpb3":                     3e-12,    # observed 2.69e-13
    "fr_N20_wpb3_w":                   4e-13,    # observed 3.30e-14
    "fr_N20_wpb4":                     3e-12,    # observed 2.69e-13
    "fr_N20_wpb4_w":                   4e-13,    # observed 3.30e-14
    "fr_N32_w":                        8e-12,    # observed 7.40e-13
    "fr_N63":                          6e-12,    # observed 5.37e-13
    "fr_N64":                          5e-12,    # observed 4.09e-13
    "fr_N8_wpb3":                      2e-12,    # observed 1.08e-13
    "fr_N8_wpb3_w":                    7e-13,    # observed 6.02e-14
    "fr_N8_wpb4":                      2e-12,    # observed 1.08e-13
    "fr_N8_wpb4_w":                    7e-13,    # observed 6.02e-14
    "fr_N95_w":                        4e-10,    # observed 3.02e-11
    "fr_tpp_N20":                      2e-11,    # observed 1.30e-12
    "fr_tpp_N40_w":                    2e-10,    # observed 1.49e-11
    "fr_tpp_N8_w":                     3e-12,    # observed 2.32e-13
    "fused_N8":                        3e-13,    # observed 2.18e-14
    "fused_N8_w":                      2e-11,    # observed 1.10e-12
    "long_N40":                        5e-13,    # observed 4.17e-14
    "long_N40_w":                      9e-13,    # observed 8.32e-14
    "long_N80":                        5e-13,    # observed 4.30e-14
    "long_N80_w":                      9e-13,    # observed 8.55e-14
    "pipeline_N8":                     3e-13,    # observed 2.14e-14
    "pipeline_N8_w":                   2e-11,    # observed 1.10e-12
    "records_device":                  4e-13,    # observed 3.22e-14
    "xy_N20":                          2e-12,    # observed 1.73e-13
    "xy_N3":                           2e-12,    # observed 1.75e-13
    "xy_N31_w":                        1e-12,    # observed 9.88e-14
    "xy_N32":                          2e-13,    # observed 1.31e-14
    "xy_N63_w":                        2e-13,    # observed 1.89e-14
    "xy_N64_w":                        3e-13,    # observed 2.69e-14
    "xy_N8_w":                         6e-11,    # observed 5.81e-12
    "xy_N95":                          3e-13,    # observed 2.34e-14
    "xy_tpp_N20_w":                    2e-09,    # observed 1.21e-10
    "xy_tpp_N40":                      4e-12,    # observed 3.07e-13
    "xy_tpp_N8":                       9e-11,    # observed 8.36e-12
    "const_acceleration_limits_team":  8e-12,    # observed 7.45e-13
    "const_acceleration_limits_tpp":   4e-11,    # observed 3.18e-12
    "const_coarse_step_team":          2e-12,    # observed 1.12e-13
    "const_coarse_step_tpp":           3e-12,    # observed 2.37e-13
    "const_fine_step_team":            2e-12,    # observed 1.61e-13
    "const_fine_step_tpp":             7e-12,    # observed 6.69e-13
    "const_rear_axle_reference_team":  4e-12,    # observed 3.32e-13
    "const_rear_axle_reference_tpp":   7e-11,    # observed 6.79e-12
    "const_reverse_and_fast_team":     4e-12,    # observed 3.01e-13
    "const_reverse_and_fast_tpp":      7e-12,    # observed 6.80e-13
    "const_steering_limits_team":      2e-12,    # observed 1.20e-13
    "const_steering_limits_tpp":       4e-11,    # observed 3.28e-12
    "const_tol_1e-6_team":             2e-11,    # observed 1.38e-12
    "const_tol_1e-6_tpp":              6e-11,    # observed 5.55e-12
    "const_wheelbase_team":            3e-12,    # observed 2.63e-13
    "const_wheelbase_tpp":             2e-11,    # observed 1.48e-12
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
        print("observed %-34s %.2e  (bar %.0e)" % (row, OBSERVED[row], bar(row)))


@pytest.fixture(scope="module")
def capi():
    from mkz_mpc_path_follower_b200 import capi as c
    c.lib()
    return c


class frenet_block_size(object):
    """MPCB200_FRENET_WPB for the handles created inside (it is read only when a handle is created); restored on exit."""

    def __init__(self, wpb):
        self.wpb, self.keep = wpb, None

    def __enter__(self):
        self.keep = os.environ.get("MPCB200_FRENET_WPB")
        if self.wpb is not None:
            os.environ["MPCB200_FRENET_WPB"] = str(self.wpb)

    def __exit__(self, *exc):
        if self.keep is None:
            os.environ.pop("MPCB200_FRENET_WPB", None)
        else:
            os.environ["MPCB200_FRENET_WPB"] = self.keep


def gpu_solve(capi, case, max_iter, tpp, wpb=None):
    """The case through the C ABI on a handle built with the case's constants and cap."""
    with frenet_block_size(wpb):
        s = (capi.FrenetSolver if case.model else capi.Solver)(case.N, max_iter=max_iter, **case.consts)
    try:
        s.set_large_batch_path(1 if tpp else 0)
        state, ref, v_des, u_prev = case.inputs
        g = s.solve_batch(state, ref, u_prev, v_des=v_des, warm=case._warm(), want_traj=True, weights=case.rows)
    finally:
        s.close()
    return g


def check_case(capi, row, case, tpp, wpb=None, ks=KS):
    for k in ks:
        o, g = case.oracle(k), gpu_solve(capi, case, k, tpp, wpb)
        assert np.array_equal(o["status"], g["status"]), (row, k, o["status"], g["status"])
        assert (o["status"] == 3).any(), (row, k)
        observe(row, iterate_error(o, g))
    o, g = case.oracle(200), gpu_solve(capi, case, 200, tpp, wpb)
    assert np.array_equal(o["status"], g["status"]), (row, o["status"], g["status"])
    short = o["iters"] <= FULL_ITERS
    assert short.any() and np.array_equal(o["iters"][short], g["iters"][short]), (row, o["iters"], g["iters"])
    ok = o["status"] == 0
    assert ok.mean() >= 0.5
    assert np.abs(o["u0"] - g["u0"])[ok].max() <= U_BAR


@pytest.mark.parametrize("row", list(SOLVE_ROWS))
def test_solve_kernel_iterates(capi, oracle, row):
    kernel, model, N, B, layout, weighted, warm, wpb = SOLVE_ROWS[row]
    case = Case(oracle, model, N, B, weighted=weighted, warm=warm)
    check_case(capi, row, case, layout == "tpp", wpb)


@pytest.mark.parametrize("tpp", [False, True], ids=["team", "tpp"])
@pytest.mark.parametrize("name", list(CONSTANT_SETS))
def test_model_constants(capi, oracle, name, tpp):
    """The constant sets of the CPU sweep (test_iterates_emu.py) at N = 8, one warp per problem (mpc_solve_kernel<0>) and one
    thread per problem (mpc_solve_tpp_kernel<0, 0>), each against the oracle built with the same constants."""
    case = Case(oracle, 0, 8, 96 if tpp else 24, **CONSTANT_SETS[name])
    check_case(capi, "const_%s_%s" % (name, "tpp" if tpp else "team"), case, tpp, ks=(2, 5))


def test_records_and_device_pointers(capi, oracle):
    """The unpacked solve path (B = 96 > 64, one warp per problem): mpcb200_solve_batch_records with host pointers and
    mpcb200_solve_batch with device pointers return the oracle's capped iterate, and the same one as mpcb200_solve_batch."""
    import torch
    N, B, k = 20, 96, 3
    case = Case(oracle, 0, N, B, warm=True)
    state, ref, v_des, u_prev = case.inputs
    o = case.oracle(k)
    s = capi.Solver(N, max_iter=k)
    s.set_large_batch_path(0)
    g = s.solve_batch(state, ref, u_prev, v_des=v_des, warm=case._warm(), want_traj=True)
    observe("records_device", iterate_error(o, g))
    warm = case._warm()
    rec = s.solve_batch_records(state, ref, u_prev, v_des=v_des, warm=warm)        # warm: in the start, out the iterate
    assert np.array_equal(warm, g["traj"]) and np.array_equal(rec[:, 0:2], g["u0"])
    dev = torch.device("cuda", 0)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device=dev)
    u0 = torch.empty((B, 2), dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    traj = torch.empty((B, 6 * N + 4), dtype=torch.float64, device=dev)
    dwarm = t(case.warm)
    s.solve_batch_device(B, t(state), t(ref), t(u_prev), u0, v_des=t(v_des), warm=dwarm, status=status, traj=traj)
    torch.cuda.synchronize()
    assert np.array_equal(traj.cpu().numpy(), g["traj"]) and np.array_equal(dwarm.cpu().numpy(), g["traj"])
    assert np.array_equal(u0.cpu().numpy(), g["u0"]) and np.array_equal(status.cpu().numpy(), o["status"])
    s.close()


def test_module_load_seed_is_capped_like_the_oracle(oracle):
    """A rollout's first solve starts from the module-load solution, which the library and mpc_oracle_module_load_solution both
    solve under the handle's cap: at max_iter = 3 that seed is a 3-iteration iterate, not the converged solution.  (The rollout
    rows below would differ from the first period on if the two capped it differently.)"""
    capped = oracle.module_load_solution(oracle.default_cfg(8, max_iter=3))
    full = oracle.module_load_solution(oracle.default_cfg(8))
    assert np.abs(capped - full).max() > 1e-3


@pytest.mark.parametrize("row", list(ROLLOUT_ROWS))
def test_rollout_kernel_iterates(capi, oracle, row):
    """Closed loop with max_iter = 3 in every period (each period's solve stops at an interior iterate, so a wrong step shows in
    the published command) against the oracle's closed loop with the same cap, vehicle by vehicle."""
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    kernel, N, weighted, pipeline = ROLLOUT_ROWS[row]
    T, k = 6, 3
    g = GPSRefTrajectory(mat_filename=1, traj_horizon=N, traj_dt=0.2)
    rng = np.random.default_rng(N)
    poses = np.array([g.trajectory[j, [4, 5, 3]] + rng.normal(scale=[0.3, 0.3, 0.03]) for j in (0, 900, 2500, 4000, 5200)])
    B = poses.shape[0]
    rows = weight_rows(B, 8, seed=N) if weighted else None
    s = capi.Solver(N, max_iter=k)
    s.set_path(0, g.trajectory)
    s.set_large_batch_path(1 if pipeline else 0)
    out = s.rollout(poses, np.zeros(B, dtype=np.int32), T, weights=rows)
    s.close()
    path, keep = oracle.make_path(g.trajectory)
    capped = 0
    for v in range(B):
        olog = oracle.closed_loop(oracle.default_cfg(N, max_iter=k, weights=None if rows is None else rows[v]), path, poses[v], T)
        glog = out["log"][:, v, :]
        assert np.array_equal(glog[:, 6], olog[:, 6]) and np.array_equal(glog[:, 7], olog[:, 7]), (row, v, glog[:, 6:], olog[:, 6:])
        capped += (olog[:, 6] == 3).sum()
        observe(row, (np.abs(glog[:, 0:6] - olog[:, 0:6]) / np.maximum(1.0, np.abs(olog[:, 0:6]))).max())
    assert capped >= T * (B - 1)       # interior iterates in (almost) every period; a vehicle near the end of the path may stop
