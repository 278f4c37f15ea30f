"""Tracking metrics of closed-loop rollouts accumulated on the device (mpcb200_rollout_metrics / _frenet_metrics): what they cost
and what they save.

    python tools/rollout_metrics_bench.py [--out profiles/r04_logs/rollout_metrics_bench.log] [--reps 5] [--host-periods 500]

1. Overhead: the same rollout with and without metrics, alternated --reps times after one warm-up round, kernel time from CUDA
   events (stats()["kernel_ms"]); the default fused / per-period rule picks the path (the launch count shows which).  Logs of the
   two calls are compared bit for bit.
2. Scoring a tuning sweep, the shape of tools/weights_bench.py section 3 (1,024 weight rows x 16 start poses = 16,384 vehicles x
   500 periods, N = 8), wall time of both ways:
     a. rollout_w + the log back to the host + closed_loop.tracking_metrics on the host (its brute-force nearest-sample search),
        timed over the first --host-periods periods of the log and scaled linearly to all of them when that is fewer;
     b. rollout_metrics without a log.
   The host metrics of the scored periods are compared with the device's of a metrics call over the same periods.
The card's name and power limit head the log."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mkz_mpc_path_follower_b200 import capi, closed_loop  # noqa: E402
from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory  # noqa: E402

W_XY = np.array([9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0])


def fleet(trajs, B, seed, lead=2000):
    """B start poses near random samples of paths 1-3 (at least `lead` samples before the end), path ids 0..2"""
    rng = np.random.default_rng(seed)
    pid = (np.arange(B) % 3).astype(np.int32)
    poses = np.empty((B, 3))
    for v in range(B):
        tr = trajs[pid[v]].trajectory
        j = int(rng.integers(0, tr.shape[0] - lead))
        poses[v] = tr[j, [4, 5, 3]] + rng.normal(scale=[0.3, 0.3, 0.03])
    return poses, pid


def solver(frenet, N, trajs):
    s = capi.FrenetSolver(N) if frenet else capi.Solver(N)
    for i, g in enumerate(trajs):
        s.set_path(i, g.trajectory)
    return s


def overhead(out, reps, trajs):
    out("## 1. overhead of the metrics (kernel_ms, CUDA events; without vs with, alternated)")
    cases = [("XY N=8 16384x500", False, 8, 16384, 500), ("XY N=8 2048x500", False, 8, 2048, 500),
             ("XY N=40 512x100", False, 40, 512, 100), ("Frenet N=8 16384x200", True, 8, 16384, 200),
             ("Frenet N=8 2048x200", True, 8, 2048, 200)]
    for name, frenet, N, B, T in cases:
        s = solver(frenet, N, trajs)
        poses, pid = fleet(trajs, B, seed=B + N)
        t = {False: [], True: []}
        launches = {}
        res = {}
        for r in range(reps + 1):
            for met in (False, True):
                res[met] = s.rollout(poses, pid, T, metrics=met)
                if r:   # the first round warms both up
                    t[met].append(s.stats()["kernel_ms"])
                launches[met] = s.stats()["kernel_launches"]
        same = np.array_equal(res[False]["log"], res[True]["log"], equal_nan=True) and np.array_equal(res[False]["final_state"], res[True]["final_state"])
        m0, m1 = np.median(t[False]), np.median(t[True])
        out("%-22s without %s ms (median %.2f, %d launches)" % (name, " ".join("%.2f" % x for x in t[False]), m0, launches[False]))
        out("%-22s with    %s ms (median %.2f, %d launches)  ratio %.4f  spread without %.2f %%  log and final bit-identical: %s"
            % ("", " ".join("%.2f" % x for x in t[True]), m1, launches[True], m1 / m0, 100 * (max(t[False]) - min(t[False])) / m0, same))


def sweep(out, trajs, host_periods):
    out("## 2. scoring a tuning sweep: 1,024 weight rows x 16 start poses (paths 1-3) = 16,384 vehicles x 500 periods, N = 8")
    N, T, R, P = 8, 500, 1024, 16
    s = solver(False, N, trajs)
    poses16, pid16 = fleet(trajs, P, seed=3)
    rng = np.random.default_rng(99)
    rows = np.where(W_XY > 0, W_XY, 1.0) * 10.0 ** rng.uniform(-1.0, 1.0, size=(R, 8))
    rows[0] = W_XY
    poses, path_of, w = np.tile(poses16, (R, 1)), np.tile(pid16, R), np.repeat(rows, P, axis=0)
    s.rollout(poses[:64], path_of[:64], 5, weights=w[:64])   # module-load solve, buffers
    s.rollout(poses[:64], path_of[:64], 5, weights=w[:64], metrics=True, want_log=False)
    hp = min(host_periods, T)
    t0 = time.perf_counter()
    r = s.rollout(poses, path_of, T, weights=w)
    t_roll = time.perf_counter() - t0
    k_roll = s.stats()["kernel_ms"]
    t0 = time.perf_counter()
    host = np.empty((R * P, 12))
    for p in range(3):
        m = path_of == p
        host[m] = closed_loop.tracking_metrics(r["log"][:hp, m, :], trajs[p].trajectory)
    t_host = time.perf_counter() - t0
    t_host_all = t_host * T / hp
    out("a. rollout_w with log: wall %.3f s (kernel %.1f ms, log %.0f MB); tracking_metrics on the host over %d of %d periods: %.1f s%s;"
        " total %.1f s" % (t_roll, k_roll, r["log"].nbytes / 1e6, hp, T, t_host,
                          "" if hp == T else " (x %d / %d = %.1f s for all periods, scaled linearly)" % (T, hp, t_host_all), t_roll + t_host_all))
    t0 = time.perf_counter()
    d = s.rollout(poses, path_of, T, weights=w, metrics=True, want_log=False)
    t_met = time.perf_counter() - t0
    st = s.stats()
    out("b. rollout_metrics without log: wall %.3f s (kernel %.1f ms, %d launches, %.1f MB back)" % (t_met, st["kernel_ms"], st["kernel_launches"], st["d2h_bytes"] / 1e6))
    out("   wall a / b: %.1fx" % ((t_roll + t_host_all) / t_met))
    dh = s.rollout(poses, path_of, hp, weights=w, metrics=True, want_log=False)["metrics"]
    exact = [0, 3, 5, 8, 9, 10, 11]
    rest = [1, 2, 4, 6, 7]
    rel = np.abs(dh[:, rest] - host[:, rest]) / np.maximum(np.abs(host[:, rest]), 1e-300)
    out("   device metrics of a %d-period call against the host's of the first %d logged periods: fields %s bit-equal: %s; max rel. "
        "difference of the others %.2e" % (hp, hp, exact, np.array_equal(dh[:, exact], host[:, exact], equal_nan=True), rel.max()))
    med = d["metrics"][:, 2].reshape(R, P).mean(axis=1)
    order = np.argsort(med)
    out("   rows ranked by mean over poses of path_err_rms [m]: best %s, module defaults (row 0) rank %d of %d"
        % (" ".join("%d:%.4f" % (i, med[i]) for i in order[:5]), int(np.nonzero(order == 0)[0][0]) + 1, R))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_logs", "rollout_metrics_bench.log"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-periods", type=int, default=500, help="periods of the log scored on the host in section 2")
    a = ap.parse_args()
    if a.reps < 1 or a.host_periods < 1:
        ap.error("--reps and --host-periods must be at least 1")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    f = open(a.out, "w")

    def out(line):
        print(line)
        f.write(line + "\n")
        f.flush()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out("# tools/rollout_metrics_bench.py on %s" % q.stdout.strip().splitlines()[0])
    trajs = [GPSRefTrajectory(mat_filename=p) for p in (1, 2, 3)]
    overhead(out, a.reps, trajs)
    sweep(out, trajs, a.host_periods)
    f.close()


if __name__ == "__main__":
    main()
