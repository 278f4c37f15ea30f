"""CPU check of the solver's path, not only its end point: the kernel sources compiled for the host (tests/emu) must return the
oracle's iterate after every capped number of iterations.

An interior-point method corrects itself: a slightly wrong Newton step (one Hessian term, one Riccati lane role, one gain) still
ends at the same KKT point after a few more line-search trials, so a check of converged solutions alone cannot see it.  The
iterate after k = 1, 2, 3, 5, 10 iterations (max_iter = k, status UserLimit) separates a correct kernel from a broken one by
orders of magnitude: with ∂²β of TeamSolver::eval_point off by 1 %, the iterate after 2 iterations at N = 8 is off by 3e-4
while the converged command is still within 1e-9 of the oracle's.

  * capped iterates: the returned trajectory against the oracle's at the same cap, relative to max(1, |traj|), bar ITER_BAR
    (measured: 1e-15 to 1.3e-12);
  * full solves: equal statuses, equal iteration counts wherever the oracle needs at most FULL_ITERS iterations, and the
    same command where the solve is Optimal;
  * both device layouts (one warp / block of warps per problem, one thread per problem), both models, the handle's weights and
    one weight row per problem (PW = 1), horizons at the one-warp edges and the 2- and 3-warp teams;
  * the model constants of mpcb200_config (dt, dt_control, L_a, L_b, the bounds, the rate limits, tol), each set against the
    oracle built with the same constants.
Long XY horizons (N > 31) start from the reference waypoints (workload.reference_start): from the all-zero start the path there is
chaotic and a rounding difference alone changes the iteration count."""
import os
import sys

import numpy as np
import pytest

from mkz_mpc_path_follower_b200 import workload as W

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

KS = (1, 2, 3, 5, 10)
ITER_BAR = 1e-10       # capped iterates, relative to max(1, |traj|)
FULL_ITERS = 60        # full solves: iteration counts must agree where the oracle needs at most this many
U_BAR = 1e-9           # full solves: |du| where Optimal

W_XY = np.array([9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0])   # MKZMPCPathFollower.jl:51-59
W_FRENET = np.array([9.0, 10.0, 0.5, 100.0, 1000.0, 0.0, 0.0])     # MKZMPCPathFollowerFrenet.jl:51-58

# the model constants a user with another vehicle or another time step changes (mpcb200_config)
CONSTANT_SETS = {
    "wheelbase": dict(L_a=1.5, L_b=1.2),
    "rear_axle_reference": dict(L_a=0.0),
    "fine_step": dict(dt=0.1, dt_control=0.05),
    "coarse_step": dict(dt=0.3, dt_control=0.3),
    "reverse_and_fast": dict(v_min=-2.0, v_max=12.0),
    "acceleration_limits": dict(a_max=3.0, a_dmax=0.5),
    "steering_limits": dict(steer_max=1.2, steer_dmax=2.0),
    "tol_1e-6": dict(tol=1e-6),
}


@pytest.fixture(autouse=True)
def _race_check():
    """Every emulated run is also a shared-memory race check (as in test_emu_parity.py)."""
    import emu as E
    E.race_check(True)
    yield
    assert E.race_count() == 0


def weight_rows(B, n, seed):
    """Distinct rows, log-uniform in [0.3x, 3x] the module defaults (entries whose default is 0 around 1), row 0 the defaults."""
    rng = np.random.default_rng(seed)
    base = W_XY if n == 8 else W_FRENET
    rows = np.where(base > 0, base, 1.0) * 10.0 ** rng.uniform(-0.5, 0.5, size=(B, n))
    rows[0] = base
    return rows


class Case(object):
    """One configuration of the matrix: model (0 XY, 1 Frenet), horizon, batch, layout, weights, start point, model constants."""

    def __init__(self, oracle, model, N, B, tpp=False, weighted=False, warm=False, **consts):
        self.O, self.model, self.N, self.tpp, self.consts = oracle, model, N, tpp, consts
        dt = consts.get("dt", 0.2)
        if model:
            b = W.make_frenet_batch(B, N, dt=dt)
            self.inputs = (b["state"], b["kpoly"], b["v_des"], b["u_prev"])
        else:
            b = W.make_batch(B, N, dt=dt)
            self.inputs = (b["state"], b["ref"], b["v_des"], b["u_prev"])
        self.warm = W.reference_start(b, N) if warm else None
        self.rows = weight_rows(B, 7 if model else 8, seed=1000 * model + N) if weighted else None

    def cfg(self, max_iter, row=None):
        if self.model:
            w = None if row is None else np.concatenate([[0.0], row])
            return self.O.default_cfg_frenet(self.N, weights=w, max_iter=max_iter, **self.consts)
        return self.O.default_cfg(self.N, weights=row, max_iter=max_iter, **self.consts)

    def _warm(self):
        return None if self.warm is None else self.warm.copy()

    def oracle(self, max_iter):
        solve = self.O.solve_batch_frenet if self.model else self.O.solve_batch
        if self.rows is None:
            return solve(self.cfg(max_iter), *self.inputs, warm=self._warm(), want_traj=True, n_threads=4)
        warm = self._warm()
        outs = [solve(self.cfg(max_iter, self.rows[j]), *[a[j:j + 1] for a in self.inputs],
                      warm=None if warm is None else warm[j:j + 1].copy(), want_traj=True, n_threads=1) for j in range(len(self.rows))]
        return {k: np.concatenate([o[k] for o in outs]) for k in ("u0", "status", "iters", "traj")}

    def emulated(self, max_iter):
        import emu as E
        import emu_weights as EW
        kc = E.kcfg_from_oracle(self.cfg(max_iter))
        if self.rows is not None:
            fn = EW.solve_batch_frenet_w if self.model else EW.solve_batch_w
            return fn(kc, *self.inputs, self.rows, warm=self._warm(), want_traj=True, tpp=self.tpp, slots=5)
        if self.model:
            return E.solve_batch_frenet(kc, *self.inputs, warm=self._warm(), want_traj=True, tpp=self.tpp, slots=5)
        if self.tpp:
            return E.solve_batch_tpp(kc, *self.inputs, warm=self._warm(), want_traj=True, slots=5)
        return E.solve_batch(kc, *self.inputs, warm=self._warm(), want_traj=True)


def iterate_error(o, e):
    """Largest difference of the returned trajectories, relative to max(1, |traj|); NaN stays NaN and fails every bar."""
    return (np.abs(e["traj"] - o["traj"]) / np.maximum(1.0, np.abs(o["traj"]))).max()


def check_capped(case, ks=KS):
    for k in ks:
        o, e = case.oracle(k), case.emulated(k)
        assert np.array_equal(o["status"], e["status"]), (k, o["status"], e["status"])
        assert (o["status"] == 3).any(), k          # the cap was reached: this is an interior iterate
        d = iterate_error(o, e)
        assert d <= ITER_BAR, (k, d)


def check_full(case, max_iter=200, min_optimal=0.5):
    o, e = case.oracle(max_iter), case.emulated(max_iter)
    assert np.array_equal(o["status"], e["status"]), (o["status"], e["status"])
    short = o["iters"] <= FULL_ITERS
    assert short.any()
    assert np.array_equal(o["iters"][short], e["iters"][short]), (o["iters"], e["iters"])
    ok = o["status"] == 0
    assert ok.mean() >= min_optimal
    assert np.abs(o["u0"] - e["u0"])[ok].max() <= U_BAR


XY_CASES = [(3, 12, False), (8, 12, False), (20, 8, False), (31, 4, False), (32, 3, True), (64, 3, True)]


@pytest.mark.parametrize("weighted", [False, True], ids=["handle_w", "row_w"])
@pytest.mark.parametrize("tpp", [False, True], ids=["warp", "tpp"])
@pytest.mark.parametrize("N,B,warm", XY_CASES, ids=["N%d" % c[0] for c in XY_CASES])
def test_xy_iterates_match_oracle(oracle, N, B, warm, tpp, weighted):
    """XY model: the one-warp kernel at N = 3, 8, 20, 31, the 2- and 3-warp teams at N = 32 and 64, the thread-per-problem solver
    at every one of these horizons."""
    case = Case(oracle, 0, N, B, tpp=tpp, weighted=weighted, warm=warm)
    check_capped(case)
    check_full(case)


@pytest.mark.parametrize("weighted", [False, True], ids=["handle_w", "row_w"])
@pytest.mark.parametrize("tpp", [False, True], ids=["warp", "tpp"])
@pytest.mark.parametrize("N,B", [(8, 12), (20, 8), (40, 3)], ids=["N8", "N20", "N40"])
def test_frenet_iterates_match_oracle(oracle, N, B, tpp, weighted):
    """Frenet model (every solve converges from the all-zero start here): the one-warp kernel at N = 8 and 20, the 2-warp team at
    N = 40, and the thread-per-problem solver."""
    case = Case(oracle, 1, N, B, tpp=tpp, weighted=weighted)
    check_capped(case)
    check_full(case, min_optimal=1.0)


@pytest.mark.parametrize("tpp", [False, True], ids=["warp", "tpp"])
@pytest.mark.parametrize("N,B", [(8, 12), (20, 6)], ids=["N8", "N20"])
@pytest.mark.parametrize("name", list(CONSTANT_SETS))
def test_model_constants_match_oracle(oracle, name, N, B, tpp):
    """Each set of model constants against the oracle built with the same constants: they reach the kernels through
    kcfg_finalize (bounds, rate rows, rfrac, mu_min), dtLb and the model evaluation."""
    case = Case(oracle, 0, N, B, tpp=tpp, **CONSTANT_SETS[name])
    check_capped(case, ks=(2, 5))
    check_full(case)


def test_loose_tolerance_stops_at_the_barrier_floor(oracle):
    """tol >= 1e-4 (N = 8): most solves end with MPCB200_ERROR, in the oracle and in both layouts alike.  The barrier parameter
    stops at min(tol, compl_inf_tol) / (barrier_tol_factor + 1) of the SCALED problem, while convergence asks for an UNSCALED
    complementarity <= compl_inf_tol = 1e-4; with the objective scaled by 0.02 to 0.04 (nlp_scaling_max_gradient) that floor is
    out of reach.  The step becomes tiny at mu_min and the solve stops as Ipopt 3.12 does (MonotoneMuUpdate: TINY_STEP_DETECTED
    -> Search_Direction_Becomes_Too_Small -> :Error).  At tol = 1e-5 the same problems are all Optimal.  DESIGN.md section 5."""
    import emu as E
    N, B = 8, 24
    b = W.make_batch(B, N)
    args = (b["state"], b["ref"], b["v_des"], b["u_prev"])
    for tol, n_error in ((1e-5, 0), (1e-4, 17)):
        cfg = oracle.default_cfg(N, tol=tol)
        o = oracle.solve_batch(cfg, *args, n_threads=4)
        assert (o["status"] == 4).sum() == n_error and ((o["status"] == 0) | (o["status"] == 4)).all(), tol
        kc = E.kcfg_from_oracle(cfg)
        ok = o["status"] == 0
        for e in (E.solve_batch(kc, *args), E.solve_batch_tpp(kc, *args, slots=5)):
            # the tiny-step test compares the step with machine epsilon: whether a solve stalled at the floor stops there (Error)
            # or runs on to the cap (UserLimit) depends on rounding
            assert np.array_equal(e["status"] == 0, ok) and np.isin(e["status"][~ok], (3, 4)).all(), tol
            assert np.abs(o["u0"] - e["u0"])[ok].max() <= U_BAR
    # the stop is the tiny-step exit at the barrier floor, not a line-search or restoration failure
    j = int(np.nonzero(o["status"] == 4)[0][0])
    r = oracle.solve(oracle.default_cfg(N, tol=1e-4), *[a[j] for a in args])
    d = r["diag"]
    assert d["ipopt_status"] == -3 and d["n_resto"] == 0
    assert d["mu_final"] == pytest.approx(1e-4 / 11) and d["compl_inf"] > 1e-4 and d["constr_viol"] <= 1e-12
