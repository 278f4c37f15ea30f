"""Frenet-frame batches from vehicle poses (mpcb200_solve_batch_frenet_on_path) against the host route they replace.

    python tools/frenet_on_path_bench.py [--out profiles/r07_logs/frenet_on_path_bench.log] [--reps 5]

At N = 8 and 20 and 16,384 and 65,536 poses near paths 1-3 (0.4 m, 0.05 rad off the path, window 40 m), each alternated --reps
times after one warm-up round, medians and spread:
  (a) host route: the numpy reference step of closed_loop.run_frenet (np.argmin over the path, np.interp of the path ahead every
      0.5 m, the rotation into the vehicle frame) and frenet_ref.fit_windows on the host, then one solve_batch_frenet call; wall time
      of each part;
  (b) one solve_batch_on_path call (host arrays): wall time, and kernel time from the library's CUDA events (stats()["kernel_ms"]:
      the reference kernel, the solve and the answers for unset ids);
  (c) device pointers on the caller's stream, CUDA events: solve_batch_on_path_device (three kernels) against solve_batch_device
      on the rows it returned (the solve kernel alone); the difference is the reference kernel plus on_path_invalid_kernel.
The outputs of (b) are compared bit for bit with solve_batch_frenet on its returned rows.  The card's name and power limit head
the log."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mkz_mpc_path_follower_b200 import capi, frenet_ref  # noqa: E402
from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory  # noqa: E402

WINDOW, TARGET_VEL = 40.0, 8.0


def poses(tables, B, seed):
    rng = np.random.default_rng(seed)
    path_of = (np.arange(B) % 3).astype(np.int32)
    pose = np.empty((B, 4))
    for p in range(3):
        m = path_of == p
        tr = tables[p]
        idx = rng.integers(0, tr.shape[0] - 400, m.sum())
        pose[m, :3] = tr[idx][:, [4, 5, 3]] + rng.normal(scale=[0.4, 0.4, 0.05], size=(m.sum(), 3))
    pose[:, 3] = rng.uniform(2.0, 9.0, B)
    return pose, path_of, rng.uniform(-0.05, 0.05, (B, 2))


def host_reference(tables, pose, path_of):
    """closed_loop.run_frenet's reference step for a batch: (K, state)."""
    B = pose.shape[0]
    s_fit = np.arange(0.0, WINDOW, 0.5)
    xw = np.empty((B, s_fit.size)); yw = np.empty_like(xw)
    for b in range(B):
        tr = tables[path_of[b]]
        i = int(np.argmin((tr[:, 4] - pose[b, 0]) ** 2 + (tr[:, 5] - pose[b, 1]) ** 2))
        sq = tr[i, 6] + s_fit
        dx = np.interp(sq, tr[:, 6], tr[:, 4]) - pose[b, 0]; dy = np.interp(sq, tr[:, 6], tr[:, 5]) - pose[b, 1]
        c, s_ = np.cos(pose[b, 2]), np.sin(pose[b, 2])
        xw[b] = c * dx + s_ * dy; yw[b] = -s_ * dx + c * dy
    t1 = time.perf_counter()
    K, psi0 = frenet_ref.fit_windows(xw, yw, WINDOW)
    state = np.column_stack([np.zeros(B), -(-np.sin(psi0) * xw[:, 0] + np.cos(psi0) * yw[:, 0]), -psi0, pose[:, 3]])
    return K, state, t1


def med(v):
    v = np.asarray(v)
    return np.median(v), 100.0 * (v.max() - v.min()) / np.median(v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_logs", "frenet_on_path_bench.log"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    f = open(a.out, "w")

    def out(line):
        print(line, flush=True)
        f.write(line + "\n"); f.flush()

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out("# GPU: %s" % q.stdout.strip().splitlines()[0])
    out("# frenet_on_path_bench: window %g m, target_vel %g, medians of %d alternated runs (spread = (max - min) / median)"
        % (WINDOW, TARGET_VEL, a.reps))
    tables = [GPSRefTrajectory(mat_filename=p).trajectory for p in (1, 2, 3)]
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()   # (the legacy default stream has handle 0, which set_stream takes as "the handle's own stream")
    for N in (8, 20):
        s = capi.FrenetSolver(N)
        for p in range(3):
            s.set_path(p, tables[p])
        s.set_stream(stream.cuda_stream)
        for B in (16384, 65536):
            pose, path_of, u_prev = poses(tables, B, seed=B + N)
            v_des = np.full(B, TARGET_VEL)
            tp = {k: torch.from_numpy(x).to(dev) for k, x in (("pose", pose), ("path_of", path_of), ("u_prev", u_prev))}
            d = {k: torch.empty(sh, dtype=dt, device=dev) for k, sh, dt in (("u0", (B, 2), torch.float64), ("k", (B, 4), torch.float64),
                                                                          ("st", (B, 4), torch.float64), ("status", (B,), torch.int32))}
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            T = {k: [] for k in ("a_ref", "a_fit", "a_solve", "b_wall", "b_kernel", "c_call", "c_solve")}
            same = True
            torch.cuda.set_stream(stream)
            for r in range(a.reps + 1):
                # (a) host route (one pass of the numpy loop per rep: it is the slow part and needs no more samples)
                t0 = time.perf_counter()
                K, state, t1 = host_reference(tables, pose, path_of)
                t2 = time.perf_counter()
                s.solve_batch(state, K, u_prev, v_des=v_des)
                t3 = time.perf_counter()
                # (b) one call, host arrays
                t4 = time.perf_counter()
                g = s.solve_batch_on_path(pose, path_of, u_prev, window=WINDOW, target_vel=TARGET_VEL, want_traj=True, want_ref=True)
                t5 = time.perf_counter()
                kms = s.stats()["kernel_ms"]
                # (c) device pointers: the call, then the solve alone on its rows
                vd = torch.full((B,), TARGET_VEL, dtype=torch.float64, device=dev)
                torch.cuda.synchronize()
                e0.record(stream)
                s.solve_batch_on_path_device(B, tp["pose"], tp["path_of"], tp["u_prev"], d["u0"], window=WINDOW, target_vel=TARGET_VEL,
                                             status=d["status"], k_coeffs_out=d["k"], state_out=d["st"])
                e1.record(stream); torch.cuda.synchronize()
                c_call = e0.elapsed_time(e1)
                e0.record(stream)
                s.solve_batch_device(B, d["st"], d["k"], tp["u_prev"], d["u0"], v_des=vd, status=d["status"])
                e1.record(stream); torch.cuda.synchronize()
                c_solve = e0.elapsed_time(e1)
                if r == 0:
                    o = s.solve_batch(g["state"], g["k_coeffs"], u_prev, v_des=v_des, want_traj=True)
                    same = all(np.array_equal(g[k], o[k]) for k in ("u0", "cost", "status", "iters", "traj"))
                    kd = np.abs(g["k_coeffs"] - K).max() / np.abs(K).max()
                    conv = (g["status"] == 0).mean()
                    continue
                for k, v in (("a_ref", t1 - t0), ("a_fit", t2 - t1), ("a_solve", t3 - t2), ("b_wall", t5 - t4)):
                    T[k].append(1e3 * v)
                T["b_kernel"].append(kms); T["c_call"].append(c_call); T["c_solve"].append(c_solve)
            m = {k: med(v) for k, v in T.items()}
            a_total = m["a_ref"][0] + m["a_fit"][0] + m["a_solve"][0]
            out("N=%-2d B=%-6d (a) host route %.1f ms = search+resample %.1f (%.1f us/problem, spread %.0f %%) + fit_windows %.1f + "
                "solve_batch_frenet %.2f (spread %.1f %%)" % (N, B, a_total, m["a_ref"][0], 1e3 * m["a_ref"][0] / B, m["a_ref"][1],
                                                          m["a_fit"][0], m["a_solve"][0], m["a_solve"][1]))
            out("           (b) solve_batch_on_path wall %.2f ms (spread %.1f %%), kernel %.3f ms (spread %.1f %%); %.0fx the host route"
                % (m["b_wall"][0], m["b_wall"][1], m["b_kernel"][0], m["b_kernel"][1], a_total / m["b_wall"][0]))
            out("           (c) device call %.3f ms (spread %.1f %%), solve kernel alone %.3f ms (spread %.1f %%): reference + invalid-id "
                "kernels %.3f ms = %.1f %% of the call" % (m["c_call"][0], m["c_call"][1], m["c_solve"][0], m["c_solve"][1],
                                                          m["c_call"][0] - m["c_solve"][0], 100.0 * (m["c_call"][0] - m["c_solve"][0]) / m["c_call"][0]))
            out("           outputs of (b) bit-identical to solve_batch_frenet on its rows: %s; Optimal %.4f; max |K - K_host| / max |K_host| %.1e"
                % (same, conv, kd))
        s.close()
    f.close()


if __name__ == "__main__":
    main()
