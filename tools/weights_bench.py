"""Per-problem cost weights on the GPU (mpcb200_solve_batch_w / _frenet_w / mpcb200_rollout_w): what they cost and what they buy.

    python tools/weights_bench.py [--out profiles/r03_logs/weights_bench.log] [--reps 5]

1. Overhead: the weighted call with every row equal to the handle's weights against the unweighted call, alternated --reps times,
   kernel time from CUDA events (stats()["kernel_ms"]): N = 20, 65,536 cold problems (warp layout); N = 8, 262,144 (thread layout);
   Frenet N = 20, 65,536 (thread layout).
2. Open-loop sweep: 65,536 problems at N = 20, rows log-uniform in [0.1x, 10x] the module defaults (seeded); converged solves/s,
   iteration distribution, a 4,096-problem sample against the oracle with each problem's own weights.
3. Closed-loop tuning sweep: 1,024 weight rows x 16 start poses on paths 1-3 = 16,384 vehicles x 500 control periods in one
   rollout_w call; rows ranked by median path error (closed_loop.path_errors).  For comparison 16 of the settings as sequential
   set_cost + rollout calls of 256 vehicles each, extrapolated to 1,024 settings.
The card's name and power limit head the log."""
import argparse
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mkz_mpc_path_follower_b200 import capi, closed_loop, workload as W  # noqa: E402
from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory  # noqa: E402

W_XY = np.array([9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0])
W_FRENET = np.array([9.0, 10.0, 0.5, 100.0, 1000.0, 0.0, 0.0])


def log_uniform_rows(B, base, seed):
    """rows log-uniform in [0.1x, 10x] the defaults; entries whose default is 0 (cv, ca, cd) around 1 instead"""
    rng = np.random.default_rng(seed)
    return np.where(base > 0, base, 1.0) * 10.0 ** rng.uniform(-1.0, 1.0, size=(B, base.size))


def overhead(out, reps):
    out("## 1. overhead at equal weights (kernel_ms, CUDA events; unweighted vs weighted, alternated)")
    cases = [("XY N=20 B=65536 warp layout", False, 20, 65536), ("XY N=8 B=262144 thread layout", False, 8, 262144),
             ("Frenet N=20 B=65536 thread layout", True, 20, 65536)]
    for name, frenet, N, B in cases:
        s = capi.FrenetSolver(N) if frenet else capi.Solver(N)
        b = W.make_frenet_batch(B, N) if frenet else W.make_batch(B, N)
        ref = b["kpoly"] if frenet else b["ref"]
        rows = np.tile(W_FRENET if frenet else W_XY, (B, 1))
        t = {False: [], True: []}
        res = {}
        for r in range(reps + 1):
            for weighted in (False, True):
                g = s.solve_batch(b["state"], ref, b["u_prev"], v_des=b["v_des"], weights=rows if weighted else None)
                if r:   # the first round warms both up
                    t[weighted].append(s.stats()["kernel_ms"])
                res[weighted] = g
        same = all(np.array_equal(res[False][k], res[True][k]) for k in ("u0", "cost", "status", "iters"))
        mu, mw = np.median(t[False]), np.median(t[True])
        out("%-36s unweighted %s ms (median %.3f)" % (name, " ".join("%.3f" % x for x in t[False]), mu))
        out("%-36s weighted   %s ms (median %.3f)  ratio %.4f  spread of unweighted %.2f %%  outputs bit-identical: %s"
            % ("", " ".join("%.3f" % x for x in t[True]), mw, mw / mu, 100 * (max(t[False]) - min(t[False])) / mu, same))


def open_loop(out, oracle):
    out("## 2. open-loop sweep: 65,536 problems, N = 20, one weight row each")
    N, B = 20, 65536
    s = capi.Solver(N)
    b = W.make_batch(B, N)
    rows = log_uniform_rows(B, W_XY, seed=2026)
    s.solve_batch(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"], weights=rows)
    t0 = time.perf_counter()
    g = s.solve_batch(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"], weights=rows)
    wall = time.perf_counter() - t0
    k = s.stats()["kernel_ms"]
    conv = int((g["status"] == 0).sum())
    out("kernel %.2f ms, call %.2f ms; converged %d / %d; %.3g converged solves/s (kernel time)" % (k, 1e3 * wall, conv, B, conv / (k * 1e-3)))
    it = g["iters"]
    out("iterations: min %d  p10 %d  p50 %d  p90 %d  p99 %d  max %d" % tuple([it.min()] + [int(np.percentile(it, q)) for q in (10, 50, 90, 99)] + [it.max()]))
    out("status counts: %s" % {int(v): int((g["status"] == v).sum()) for v in np.unique(g["status"])})
    idx = np.random.default_rng(7).choice(B, 4096, replace=False)

    def one(j):
        cfg = oracle.default_cfg(N, weights=rows[j], tol=s.cfg.tol, max_iter=s.cfg.max_iter)
        return oracle.solve_batch(cfg, b["state"][j:j + 1], b["ref"][j:j + 1], b["v_des"][j:j + 1], b["u_prev"][j:j + 1])
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        o = list(ex.map(one, idx))
    ost = np.array([x["status"][0] for x in o]); ou = np.array([x["u0"][0] for x in o]); oc = np.array([x["cost"][0] for x in o])
    ok = (ost == 0) & (g["status"][idx] == 0)
    out("oracle sample of 4096: status mismatches %d; both converged %d; max |du| %.2e; max rel cost %.2e"
        % (int((ost != g["status"][idx]).sum()), int(ok.sum()), np.abs(ou - g["u0"][idx])[ok].max(),
           (np.abs(oc - g["cost"][idx]) / np.maximum(1.0, np.abs(oc)))[ok].max()))


def closed_loop_sweep(out):
    out("## 3. closed-loop tuning sweep: 1,024 weight rows x 16 start poses (paths 1-3) = 16,384 vehicles x 500 periods")
    N, T, R, P = 8, 500, 1024, 16
    trajs = [GPSRefTrajectory(mat_filename=p) for p in (1, 2, 3)]
    s = capi.Solver(N)
    for i, g in enumerate(trajs):
        s.set_path(i, g.trajectory)
    rng = np.random.default_rng(3)
    pose_list, pid_list = [], []
    for q in range(P):
        pid = q % 3
        tr = trajs[pid].trajectory
        j = int(rng.integers(0, tr.shape[0] - 2000))
        pose_list.append(tr[j, [4, 5, 3]] + rng.normal(scale=[0.3, 0.3, 0.03]))
        pid_list.append(pid)
    rows = log_uniform_rows(R, W_XY, seed=99)
    rows[0] = W_XY
    poses = np.tile(np.array(pose_list), (R, 1))           # vehicle v = row v // P, pose v % P
    path_of = np.tile(np.array(pid_list, dtype=np.int32), R)
    w = np.repeat(rows, P, axis=0)
    s.rollout(poses[:64], path_of[:64], 5, weights=w[:64])   # module-load solve, buffers
    t0 = time.perf_counter()
    r = s.rollout(poses, path_of, T, weights=w)
    wall = time.perf_counter() - t0
    st = s.stats()
    out("rollout_w: wall %.3f s, kernel %.1f ms, %d launches" % (wall, st["kernel_ms"], st["kernel_launches"]))
    err = np.zeros((T, R * P))
    for pid in range(3):
        m = path_of == pid
        err[:, m] = closed_loop.path_errors(r["log"][:, m, :], trajs[pid].trajectory)
    med = np.median(err.reshape(T, R, P).transpose(1, 0, 2).reshape(R, -1), axis=1)
    order = np.argsort(med)
    out("rows ranked by median path error [m] (cx cy cp cv cda cdd ca cd):")
    for rank, i in enumerate(list(order[:10]) + list(order[-3:])):
        out("  %s row %4d  median %.4f  w = %s" % ("#%-4d" % (rank + 1) if rank < 10 else "worst", i, med[i], " ".join("%.3g" % x for x in rows[i])))
    out("  module defaults (row 0): median %.4f, rank %d of %d" % (med[0], int(np.nonzero(order == 0)[0][0]) + 1, R))
    # the same settings as sequential set_cost + rollout calls, 16 settings x 256 vehicles (16 poses x 16 repeats)
    seq = capi.Solver(N)
    for i, g in enumerate(trajs):
        seq.set_path(i, g.trajectory)
    sp, spid = np.tile(np.array(pose_list), (16, 1)), np.tile(np.array(pid_list, dtype=np.int32), 16)
    seq.rollout(sp[:8], spid[:8], 5)
    t0 = time.perf_counter()
    kt = 0.0
    for i in range(16):
        seq.set_cost(rows[i])
        seq.rollout(sp, spid, T)
        kt += seq.stats()["kernel_ms"]
    wall16 = time.perf_counter() - t0
    out("sequential set_cost + rollout, 16 settings x 256 vehicles x 500: wall %.3f s, kernel %.1f ms; extrapolated to the 1,024 "
        "settings as one call per setting (%d vehicles each; a call of 16 to 256 vehicles is latency-bound, so its time is taken as "
        "that of 256): wall %.1f s" % (wall16, kt, P, wall16 / 16 * R))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_logs", "weights_bench.log"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    f = open(a.out, "w")

    def out(line):
        print(line)
        f.write(line + "\n")
        f.flush()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out("# tools/weights_bench.py on %s" % q.stdout.strip().splitlines()[0])
    from oracle import oracle as O
    O.build()
    overhead(out, a.reps)
    open_loop(out, O)
    closed_loop_sweep(out)
    f.close()


if __name__ == "__main__":
    main()
