"""Per-vehicle cost weights in the Frenet closed loop (mpcb200_rollout_frenet_w): what they cost and what they save.

    python tools/frenet_rollout_weights_bench.py [--out profiles/r06_logs/frenet_rollout_weights_bench.log] [--reps 5] [--seq-rows 16]

1. Overhead at equal rows: rollout_frenet and rollout_frenet_w with every row equal to the handle's weights, alternated --reps times
   after one warm-up round; kernel time from CUDA events (stats()["kernel_ms"]), medians and spread.  The default fused / per-period
   rule picks the form (the launch count shows which): fused at N = 8, 2,048 x 200 and N = 20, 1,024 x 100, the per-period pipeline
   at N = 8, 16,384 x 200.  The logs of the two calls are compared.
2. A Frenet tuning sweep: 1,024 weight rows (row 0 = the module defaults) x 16 start poses over paths 1-3 = 16,384 vehicles x 200
   periods, N = 8, with metrics and without a log, in one call: wall and kernel time, and the best row's median path error against
   the defaults'.  Then the same settings as sequential set_cost_frenet + rollout_frenet_metrics calls (16 vehicles each), timed
   over the first --seq-rows rows and extrapolated linearly to all 1,024; their metrics are compared with the one call's.
The card's name and power limit head the log."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mkz_mpc_path_follower_b200 import capi  # noqa: E402
from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory  # noqa: E402

W_DEFAULT = np.array([9.0, 10.0, 0.5, 100.0, 1000.0, 0.0, 0.0])   # MKZMPCPathFollowerFrenet.jl:51-58, set_cost_frenet's order


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


def solver(N, trajs):
    s = capi.FrenetSolver(N)
    for i, g in enumerate(trajs):
        s.set_path(i, g.trajectory)
    return s


def overhead(out, reps, trajs):
    out("## 1. overhead at equal rows (kernel_ms, CUDA events; rollout_frenet vs rollout_frenet_w, alternated)")
    for name, N, B, T in (("fused N=8 2048x200", 8, 2048, 200), ("fused N=20 1024x100", 20, 1024, 100),
                          ("pipeline N=8 16384x200", 8, 16384, 200)):
        s = solver(N, trajs)
        poses, pid = fleet(trajs, B, seed=B + N)
        rows = np.tile(W_DEFAULT, (B, 1))
        t = {False: [], True: []}
        launches, res = {}, {}
        for r in range(reps + 1):
            for pw in (False, True):
                res[pw] = s.rollout(poses, pid, T, weights=rows if pw else None)
                if r:   # the first round warms both up
                    t[pw].append(s.stats()["kernel_ms"])
                launches[pw] = s.stats()["kernel_launches"]
        a, b = res[False], res[True]
        same_it = np.array_equal(a["log"][:, :, 6:8], b["log"][:, :, 6:8])
        d = max(np.abs(a["log"] - b["log"]).max(), np.abs(a["final_state"] - b["final_state"]).max())
        bits = np.mean(a["log"] == b["log"])
        m0, m1 = np.median(t[False]), np.median(t[True])
        spread = lambda v: 100 * (max(v) - min(v)) / np.median(v)
        out("%-24s unweighted %s ms (median %.2f, spread %.2f %%, %d launches)"
            % (name, " ".join("%.2f" % x for x in t[False]), m0, spread(t[False]), launches[False]))
        out("%-24s weighted   %s ms (median %.2f, spread %.2f %%, %d launches)  ratio %.4f" % (
            "", " ".join("%.2f" % x for x in t[True]), m1, spread(t[True]), launches[True], m1 / m0))
        out("%-24s logs: statuses and iterations equal: %s; max |d log|, |d final| %.2e; log entries bit-identical %.4f"
            % ("", same_it, d, bits))
        dv = np.nonzero((a["log"] != b["log"]).any(axis=(0, 2)))[0]
        if len(dv):   # where the two logs part: each such vehicle's first differing period and the size of that first difference
            t0 = [int(np.nonzero((a["log"][:, v] != b["log"][:, v]).any(axis=1))[0][0]) for v in dv]
            d0 = [np.abs(a["log"][t, v] - b["log"][t, v]).max() for t, v in zip(t0, dv)]
            out("%-24s %d of %d vehicles differ; first differing period min %d median %d; size of the first difference max %.2e "
                "median %.2e; vehicles whose statuses or iterations differ: %d"
                % ("", len(dv), B, min(t0), int(np.median(t0)), max(d0), np.median(d0),
                   int((a["log"][:, :, 6:8] != b["log"][:, :, 6:8]).any(axis=(0, 2)).sum())))
        s.close()


def sweep(out, trajs, seq_rows):
    N, T, R, P = 8, 200, 1024, 16
    out("## 2. Frenet tuning sweep: %d weight rows x %d start poses (paths 1-3) = %d vehicles x %d periods, N = %d, metrics, no log"
        % (R, P, R * P, T, N))
    s = solver(N, trajs)
    poses16, pid16 = fleet(trajs, P, seed=3)
    rng = np.random.default_rng(99)
    rows = np.where(W_DEFAULT > 0, W_DEFAULT, 1.0) * 10.0 ** rng.uniform(-1.0, 1.0, size=(R, 7))
    rows[0] = W_DEFAULT
    poses, path_of, w = np.tile(poses16, (R, 1)), np.tile(pid16, R), np.repeat(rows, P, axis=0)
    s.rollout(poses, path_of, 5, weights=w, metrics=True, want_log=False)    # buffers, shared-memory setup
    t0 = time.perf_counter()
    one = s.rollout(poses, path_of, T, weights=w, metrics=True, want_log=False)
    t_one = time.perf_counter() - t0
    st = s.stats()
    out("a. one rollout_frenet_w call: wall %.3f s (kernel %.1f ms, %d launches, %.1f MB back)"
        % (t_one, st["kernel_ms"], st["kernel_launches"], st["d2h_bytes"] / 1e6))
    err = one["metrics"][:, 1].reshape(R, P)                  # path_err_mean per vehicle
    med = np.median(err, axis=1)
    order = np.argsort(med)
    out("   median over the %d poses of path_err_mean [m]: module defaults (row 0) %.4f, rank %d of %d; best rows %s"
        % (P, med[0], int(np.nonzero(order == 0)[0][0]) + 1, R, " ".join("%d:%.4f" % (i, med[i]) for i in order[:5])))
    out("   best row %d: %s" % (order[0], " ".join("%.4g" % x for x in rows[order[0]])))
    s.set_cost(rows[0])
    s.rollout(poses16, pid16, 5, metrics=True, want_log=False)   # warm-up
    t0 = time.perf_counter()
    k_ms = 0.0
    dmax = 0.0
    for r in range(seq_rows):
        s.set_cost(rows[r])
        m = s.rollout(poses16, pid16, T, metrics=True, want_log=False)["metrics"]
        k_ms += s.stats()["kernel_ms"]
        ref = one["metrics"][r * P:(r + 1) * P]
        dmax = max(dmax, float(np.nanmax(np.abs(m - ref) / np.maximum(np.abs(ref), 1e-300))))
    t_seq = time.perf_counter() - t0
    out("b. sequential set_cost_frenet + rollout_frenet_metrics (%d vehicles each): %d of %d rows timed: wall %.3f s (kernel %.1f ms)"
        % (P, seq_rows, R, t_seq, k_ms))
    out("   extrapolated to %d rows: wall %.1f s (kernel %.1f s); one call is %.1fx faster in wall time (extrapolated)"
        % (R, t_seq * R / seq_rows, k_ms * R / seq_rows / 1e3, t_seq * R / seq_rows / t_one))
    out("   metrics of the timed rows against the one call's: max relative difference %.2e" % dmax)
    s.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_logs", "frenet_rollout_weights_bench.log"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seq-rows", type=int, default=16, help="rows of the sweep timed as sequential calls in section 2")
    a = ap.parse_args()
    if a.reps < 1 or not 1 <= a.seq_rows <= 1024:
        ap.error("--reps must be at least 1 and --seq-rows in [1, 1024]")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    f = open(a.out, "w")

    def out(line):
        print(line)
        f.write(line + "\n")
        f.flush()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out("# tools/frenet_rollout_weights_bench.py on %s" % q.stdout.strip().splitlines()[0])
    trajs = [GPSRefTrajectory(mat_filename=p) for p in (1, 2, 3)]
    overhead(out, a.reps, trajs)
    sweep(out, trajs, a.seq_rows)
    f.close()


if __name__ == "__main__":
    main()
