#!/usr/bin/env python
"""Queue-order model of the on-chip solve kernel (DESIGN §6, item 3): how long a persistent grid of warps takes over a batch when
each warp pulls the next problem from a device counter, in index order or longest-predicted-first.

    python tools/queue_order_model.py                    # bench batch (b0 = 0) and the next slice (b0 = 65536), N = 20
    python tools/queue_order_model.py --cache DIR        # keep the oracle's iteration counts between runs
    python tools/queue_order_model.py --init             # also order by what the solver's initialisation computes

Per-problem iteration counts come from the oracle, which follows the kernel iterate for iterate (DESIGN 3.2).  A problem
costs 1 + iters time units on a slot; 1,776 slots (148 SMs x 12 resident warps) take problems greedily in queue order, and
the makespan is scaled so that index order on the bench batch comes to the measured 41.4 ms.  The score that orders the
queue (mpc_b200.cu: queue_key_kernel) is fitted by least squares on the first slice and judged on the second.
--init: the candidates the solver's initialisation has at hand at the pushed start point (the oracle stopped before its first
iteration: objective scaling factor, constraint violation theta_0, dual infeasibility and complementarity after the
least-squares multipliers), each alone and in a least-squares fit with the raw inputs, judged the same way.
"""
import argparse
import heapq
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SLOTS = 148 * 12
MEASURED_MS = 41.4     # mpc_solve_kernel, 65,536 problems at N = 20 from the all-zero start, one B200 (DESIGN 3.4)


def oracle_counts(B, N, b0, cache):
    from mkz_mpc_path_follower_b200 import workload
    path = os.path.join(cache, "queue_order_iters_B%d_N%d_b%d.npz" % (B, N, b0))
    b = workload.make_batch(B, N, b0=b0)
    if os.path.exists(path):
        it = np.load(path)["iters"]
    else:
        from oracle import oracle as O
        O.build()
        r = O.solve_batch(O.default_cfg(N, max_iter=200), b["state"], b["ref"], b["v_des"], b["u_prev"], n_threads=os.cpu_count() or 1)
        it = r["iters"]
        np.savez(path, iters=it)
    return b, it.astype(np.float64)


def init_quantities(b, N, b0, cache):
    """(obj_scale, theta_0, dual_inf_0, compl_inf_0) per problem: the oracle's diagnostics with max_iter = 0."""
    path = os.path.join(cache, "queue_order_init_B%d_N%d_b%d.npy" % (len(b["v_des"]), N, b0))
    if not os.path.exists(path):
        from oracle import oracle as O
        O.build()
        cfg = O.default_cfg(N, max_iter=0)
        out = np.empty((len(b["v_des"]), 4))
        for j in range(len(out)):
            d = O.solve(cfg, b["state"][j], b["ref"][j], b["v_des"][j], b["u_prev"][j])["diag"]
            out[j] = (d["obj_scale"], d["constr_viol"], d["dual_inf"], d["compl_inf"])
        np.save(path, out)
    return np.load(path)


def makespan(costs, slots=SLOTS):
    """Greedy list schedule: the next problem in queue order goes to the slot that frees first."""
    h = [0.0] * min(slots, max(1, len(costs)))
    for c in costs:
        heapq.heappush(h, heapq.heappop(h) + 1.0 + c)
    return max(h)


def features(state, ref, u_prev):
    """The raw inputs queue_key_kernel reads: distance of the vehicle from the path frame's origin (log), heading change of
    the reference over the horizon, previous steering and acceleration command."""
    X, Y = state[:, 0], state[:, 1]
    turn = ref[:, 2, -1] - ref[:, 2, 0]
    return np.column_stack([np.ones(len(X)), np.log1p(np.hypot(X, Y)), np.abs(turn), np.abs(u_prev[:, 0]), u_prev[:, 1]])


def order_by(score):
    return np.argsort(-score, kind="stable")    # descending; ties in index order, as the device's stable radix sort


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--horizon", type=int, default=20)
    ap.add_argument("--cache", default=tempfile.gettempdir())
    ap.add_argument("--init", action="store_true")
    args = ap.parse_args()
    B, N = args.batch, args.horizon
    (ba, ia), (bb, ib) = oracle_counts(B, N, 0, args.cache), oracle_counts(B, N, B, args.cache)
    unit = MEASURED_MS / makespan(ia)
    Fa = features(ba["state"], ba["ref"], ba["u_prev"])
    Fb = features(bb["state"], bb["ref"], bb["u_prev"])
    coef, *_ = np.linalg.lstsq(Fa, ia, rcond=None)
    print("score = %s . [1, log1p(hypot(X, Y)), |dpsi_ref|, |d_f_prev|, acc_prev]   (fitted on b0 = 0)" % np.array2string(coef, precision=4))
    for name, b, it, F in (("bench batch, b0 = 0 (fit)", ba, ia, Fa), ("held out, b0 = %d" % B, bb, ib, Fb)):
        s = F @ coef
        r2 = 1.0 - np.var(it - s) / np.var(it)
        print("%s: iterations p50 %d, p99 %d, max %d; score R^2 %.2f" % (name, np.percentile(it, 50), np.percentile(it, 99), it.max(), r2))
        for g in (1, 2, 4, 8):
            n = len(it) // g
            row = []
            for q in (np.arange(len(it)), order_by(it), order_by(s)):
                row.append(max(makespan(it[q[(q >= r * n) & (q < (r + 1) * n)]]) for r in range(g)) * unit)
            bound = max((1.0 + it[r * n:(r + 1) * n]).sum() / SLOTS for r in range(g)) * unit
            print("  %d GPU(s), %6d problems each: index order %6.2f ms | longest first (exact counts) %6.2f | by score %6.2f (%+.1f %%) | work bound %6.2f"
                  % (g, n, row[0], row[1], row[2], 100.0 * (row[2] / row[0] - 1.0), bound))
    if args.init:
        Ia, Ib = np.log(init_quantities(ba, N, 0, args.cache)), np.log(init_quantities(bb, N, B, args.cache))
        print("initialisation quantities, one GPU, held out (b0 = %d): index order %.2f ms" % (B, makespan(ib) * unit))
        for k, name in enumerate(("objective scaling", "theta_0", "dual infeasibility", "complementarity")):
            print("  %-20s largest first %6.2f ms, smallest first %6.2f ms" % (name, makespan(ib[order_by(Ib[:, k])]) * unit,
                                                                             makespan(ib[order_by(-Ib[:, k])]) * unit))
        for name, A, Bm in (("all four (log)", np.column_stack([np.ones(B), Ia]), np.column_stack([np.ones(B), Ib])),
                            ("all four + raw inputs", np.column_stack([Fa, Ia]), np.column_stack([Fb, Ib]))):
            c, *_ = np.linalg.lstsq(A, ia, rcond=None)
            s = Bm @ c
            print("  fit of %-22s R^2 %.2f, %6.2f ms" % (name, 1.0 - np.var(ib - s) / np.var(ib), makespan(ib[order_by(s)]) * unit))


if __name__ == "__main__":
    main()
