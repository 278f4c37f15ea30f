#!/usr/bin/env python
"""bench.py -- converged MPC solves/s at batch 64K, N=20 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 5 --warmup 3
    python bench.py --impl reference ...      # CPU arm: the oracle (restated interior point, NOT Ipopt)
    python bench.py ... --dump-outputs DIR    # also the last timed step's results as DIR/*.npy, to compare two builds

A step = one pass of the hot path (cold-start solve of every problem of the batch) over one
synthetic batch: BASELINE.json configs[2], 65,536 problems per GPU at N=20 along paths 1-3
(SURVEY.md 8d).  Weak scaling: every rank solves its own contiguous 65,536-problem slice of the
counter-based stream; the only inter-GPU traffic is one NCCL all-gather of the 32 B/problem
result record.  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_RIC, F_EVAL = 1235, 310  # SURVEY.md 8(d): algorithmic flops per stage per interior-point iteration


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=65536, help="problems per GPU")
    ap.add_argument("--horizon", type=int, default=20)
    ap.add_argument("--cpu-sample", type=int, default=0, help="problems in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--sweep-batch", type=int, default=131072, help="problems per GPU and horizon of the horizon_sweep key (configs[4]: 1 M over 8 GPUs)")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs beside the headline (config1, rollout_config3, horizon_sweep, strong_64k, layouts_n8)")
    ap.add_argument("--parity", default="full", choices=["full", "sample"],
                    help="full: every problem of every rank's slice is checked against the oracle (the converged count); sample: a bounded sample")
    ap.add_argument("--rollout-vehicles", type=int, default=16384)
    ap.add_argument("--rollout-steps", type=int, default=500)
    ap.add_argument("--x0", dest="start", default="zero", choices=["zero", "rollout"],
                    help="start point: zero = the reference's start=0.0 (the metric); rollout = MPCB200_START_ROLLOUT "
                         "(opt-in; what the horizon sweep of configs[4] uses at N = 40 / 80)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (u0, cost, status, iters, restorations, "
                         "one row per problem) as DIR/<name>.npy in float64, with the problems' ids in DIR/index.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT = 64 << 20   # bytes of .npy data written by --dump-outputs


def dump_outputs(out_dir, index, arrays):
    """Writes arrays (one row per problem; index = the problems' ids in the synthetic stream) as out_dir/<name>.npy in
    float64.  When they exceed DUMP_LIMIT in all, a fixed, seeded sample of the rows is written instead."""
    index = np.asarray(index)
    n = index.shape[0]
    row_bytes = 8 * (1 + sum(int(np.prod(a.shape[1:])) for a in arrays.values()))
    rows = np.arange(n)
    if n * row_bytes > DUMP_LIMIT - 4096 * (1 + len(arrays)):     # room for the .npy headers
        k = (DUMP_LIMIT - 4096 * (1 + len(arrays))) // row_bytes
        rows = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "index.npy"), index[rows].astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(np.asarray(a)[rows], dtype=np.float64))


class ClockSampler(object):
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md): one
    `nvidia-smi -lms 100` child for the whole region, parsed when it is stopped."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        n = 0
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            n += 1
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                pass
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": n}


class NvmlClockSampler(object):
    """The same through NVML (pynvml), polled every 5 ms from a thread: the timed region is a few hundred ms, too short
    for more than a sample or two of `nvidia-smi -lms 100`.  Falls back to ClockSampler when NVML is not usable."""
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index = index
        self.fallback = None
        self.thread = None
        self.samples = []
        self.mask = 0
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
            self.fallback = ClockSampler(index)

    def _reasons(self):
        for fn in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
            f = getattr(self.nv, fn, None)
            if f is not None:
                try:
                    return int(f(self.h))
                except Exception:
                    pass
        return 0

    def _run(self):
        while not self._stop:
            try:
                self.samples.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                self.mask |= self._reasons()
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.fallback is not None:
            return self.fallback.start()
        import threading
        self._stop = False
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        if self.fallback is not None:
            return self.fallback.stop()
        self._stop = True
        self.thread.join(timeout=2)
        reasons = sorted(name for bit, name in self.BITS.items() if self.mask & bit)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(self.samples), "source": "nvml, 5 ms poll"}


def cpu_baseline(N, sample, threads, start_b0=0, start="zero", max_iter=None):
    """The oracle (restated CPU interior point, NOT Ipopt) on a bounded sample of the same workload."""
    from oracle import oracle as O
    from mkz_mpc_path_follower_b200 import workload
    O.build()
    b = workload.make_batch(sample, N, b0=start_b0)
    cfg = O.default_cfg(N, max_iter=max_iter)
    warm = O.rollout_start(cfg, b["state"], b["u_prev"]) if start == "rollout" else None
    t0 = time.perf_counter()
    r = O.solve_batch(cfg, b["state"], b["ref"], b["v_des"], b["u_prev"], warm=warm, n_threads=threads)
    dt = time.perf_counter() - t0
    conv = int((r["status"] == 0).sum())
    return conv / dt, dt, conv, r


def ipopt_probe(dump_dir=None, N=20, n_dump=256):
    """BASELINE.md 3.1: is the reference's real solver stack reachable on THIS box at run time?  Looks for `julia`, an
    `ipopt` executable and an importable `cyipopt`.  If cyipopt is there, the first n_dump problems of the bench batch
    are solved with the real Ipopt (tools/ipopt_golden.py: the oracle's NLP callbacks behind cyipopt.Problem) and dumped
    as golden vectors.  The probe itself never fails the bench."""
    import shutil
    found = {"julia": shutil.which("julia"), "ipopt": shutil.which("ipopt"), "cyipopt": False}
    try:
        import cyipopt  # noqa: F401
        found["cyipopt"] = getattr(cyipopt, "__version__", True)
    except Exception:
        pass
    if found["julia"]:
        try:
            found["julia_version"] = subprocess.check_output([found["julia"], "--version"], text=True, timeout=60).strip()
        except Exception as ex:
            found["julia_version"] = repr(ex)
    if found["cyipopt"] and dump_dir:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import ipopt_golden
            found["golden"] = ipopt_golden.dump(os.path.join(dump_dir, "ipopt_N%d.npz" % N), N, n_dump)
        except Exception as ex:
            found["golden"] = {"error": repr(ex)}
    found["reachable"] = bool(found["julia"] or found["ipopt"] or found["cyipopt"])
    return found


def run_reference(args):
    """--impl reference: the reference's CPU path.  Julia/JuMP/Ipopt cannot run here (SURVEY 8c; probed again at run
    time below), so this arm times the oracle port with every host core, one bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N = args.horizon
    cores = os.cpu_count() or 1
    sample = args.cpu_sample or max(256, 64 * cores)
    probe = ipopt_probe(os.path.join(ROOT, "gpurun_out") if os.path.isdir(os.path.join(ROOT, "gpurun_out")) else None, N)
    for _ in range(min(args.warmup, 1)):
        cpu_baseline(N, min(sample, 256), cores, start=args.start)
    t_tot, conv_tot = 0.0, 0
    for s in range(args.steps):
        v, dt, conv, r = cpu_baseline(N, sample, cores, start_b0=s * sample, start=args.start)
        t_tot += dt
        conv_tot += conv
    if args.dump_outputs:
        s = args.steps - 1
        dump_outputs(args.dump_outputs, np.arange(s * sample, (s + 1) * sample),
                     {"u0": r["u0"], "cost": r["cost"], "status": r["status"], "iters": r["iters"], "restorations": r["n_resto"]})
    val = conv_tot / t_tot
    line = {
        "impl": "reference", "metric": "converged MPC solves/sec at batch 64K, N=20", "value": val,
        "unit": "solves/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_tot / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[2]: N=%d cold-start solves along path1-3, bounded sample of %d problems/step "
                               "(problems [s*%d, (s+1)*%d) of the GPU arm's batch stream)" % (N, sample, sample, sample)},
        "cpu_baseline": {"value": val, "unit": "solves/s", "cores": cores, "kind": "port",
                         "sample": "%d problems/step x %d steps, restated CPU interior point (oracle), NOT Ipopt" % (sample, args.steps)},
        "ipopt_probe": probe,
        "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def frenet_roofline(kernel_ms, B, N):
    """HBM roofline of the thread-per-problem Frenet kernel (it streams the iterate from HBM): DRAM bytes per launch as ncu measured
    them for this very workload (profiles/dram_traffic_tpp_frenet.json), over the live kernel time, against the measured copy peak."""
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic_tpp_frenet.json")))
        if tr["problems_per_launch"] != B or tr["horizon"] != N:
            return None
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs")
        ach = tr["bytes_per_launch"] / (kernel_ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": (ach / peak) if peak else None, "traffic": tr["bytes_per_launch"],
                "traffic_source": tr["source"]}
    except Exception:
        return None


def parity_counts(g_u0, g_cost, g_status, o, ids0=0):
    """SURVEY 8(d): a solve is converged only with status Optimal AND parity with the oracle: same status,
    |du| <= 1e-5 on the first move, relative cost <= 1e-6."""
    st_eq = g_status == o["status"]
    both = (g_status == 0) & (o["status"] == 0)
    du = np.abs(g_u0 - o["u0"]).max(axis=1)
    rc = np.abs(g_cost - o["cost"]) / np.maximum(1.0, np.abs(o["cost"]))
    ok = both & (du <= 1e-5) & (rc <= 1e-6)
    bad = np.nonzero(~st_eq | (both & ~ok))[0]
    return ok, {
        "sample": int(g_status.shape[0]), "status_mismatch": int((~st_eq).sum()),
        "du_gt_1e-5": int((both & (du > 1e-5)).sum()), "relcost_gt_1e-6": int((both & (rc > 1e-6)).sum()),
        "converged_and_in_parity": int(ok.sum()), "gpu_optimal": int((g_status == 0).sum()), "oracle_optimal": int((o["status"] == 0).sum()),
        "max_abs_du": float(du[both].max()) if both.any() else None, "p999_abs_du": float(np.quantile(du[both], 0.999)) if both.any() else None,
        "mismatch_ids": [int(i) + ids0 for i in bad[:32]],
        "tolerance": "status equal, |du| <= 1e-5, |dcost| <= 1e-6 max(1, |cost|) (north_star)"}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from mkz_mpc_path_follower_b200 import capi, sharding, workload

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the solver has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N, B = args.horizon, args.batch
    cores = os.cpu_count() or 1

    def allmax(v):
        t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(vs):
        t = torch.tensor([float(v) for v in vs], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()]

    # ---- synthetic batch: this rank's contiguous slice of the problem stream
    b = workload.make_batch(B, N, b0=rank * B)
    solver = capi.Solver(N, device=local, start_mode=capi.START_ROLLOUT if args.start == "rollout" else capi.START_ZERO)
    stream = torch.cuda.Stream(device=dev)  # a real (non-NULL) stream shared by torch and the library
    torch.cuda.set_stream(stream)
    solver.set_stream(stream.cuda_stream)
    d_state = torch.from_numpy(b["state"]).to(dev)
    d_ref = torch.from_numpy(b["ref"]).to(dev)
    d_uprev = torch.from_numpy(b["u_prev"]).to(dev)
    d_vdes = torch.from_numpy(b["v_des"]).to(dev)
    d_rec = torch.empty((B, 4), dtype=torch.float64, device=dev)   # the packed 32-byte records, written by the kernel
    d_all = torch.empty((world * B, 4), dtype=torch.float64, device=dev) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step():
        flush.zero_()  # L2 flush between timed iterations (inputs are 36 MB < L2)
        solver.solve_batch_records_device(B, d_state, d_ref, d_uprev, d_rec, v_des=d_vdes)
        if world > 1:   # the one exchange step: all-gather of the 32 B/problem result record the kernel wrote
            dist.all_gather_into_tensor(d_all, d_rec)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    # kernel-only time of one step (events directly around the kernel) for the roofline
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern_ms = []
    sampler = NvmlClockSampler(local)
    sampler.start()
    barrier()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        flush.zero_()
        e0.record()
        solver.solve_batch_records_device(B, d_state, d_ref, d_uprev, d_rec, v_des=d_vdes)
        e1.record()
        if world > 1:
            dist.all_gather_into_tensor(d_all, d_rec)
        e1.synchronize()
        kern_ms.append(e0.elapsed_time(e1))
    t1.record()
    barrier()
    clocks = sampler.stop()
    total_ms = allmax(t0.elapsed_time(t1))
    km = torch.zeros(world, dtype=torch.float64, device=dev)
    km[rank] = float(np.mean(kern_ms))
    if world > 1:
        dist.all_reduce(km, op=dist.ReduceOp.SUM)
    kernel_ms_per_rank = [round(float(v), 3) for v in km.tolist()]

    u0, cost, status, iters, resto = sharding.unpack_records_np(d_rec.cpu().numpy())
    u0 = u0.copy(); cost = cost.copy()
    optimal_local = int((status == 0).sum())
    if args.dump_outputs and rank == 0:
        # the records of the last timed step: this rank's, or every rank's after the all-gather
        ru0, rcost, rstatus, riters, rresto = (sharding.unpack_records_np(d_all.cpu().numpy()) if world > 1
                                               else (u0, cost, status, iters, resto))
        dump_outputs(args.dump_outputs, np.arange(ru0.shape[0]),
                     {"u0": ru0, "cost": rcost, "status": rstatus, "iters": riters, "restorations": rresto})

    # ---- parity against the oracle on EVERY problem of this rank's slice (SURVEY 8d: converged = Optimal AND within
    # tolerance of the oracle); at one GPU this run is also the cpu_baseline (the oracle timed on the box's cores)
    from oracle import oracle as O
    O.build()
    ocfg = O.default_cfg(N, max_iter=int(solver.cfg.max_iter))
    threads = max(1, cores // world)
    n_par = B if args.parity == "full" else min(B, args.cpu_sample or max(256, 48 * cores))
    owarm = O.rollout_start(ocfg, b["state"][:n_par], b["u_prev"][:n_par]) if args.start == "rollout" else None
    tc0 = time.perf_counter()
    o = O.solve_batch(ocfg, b["state"][:n_par], b["ref"][:n_par], b["v_des"][:n_par], b["u_prev"][:n_par], warm=owarm, n_threads=threads)
    cpu_dt = time.perf_counter() - tc0
    ok, parity = parity_counts(u0[:n_par], cost[:n_par], status[:n_par], o, ids0=rank * B)
    parity["oracle_restored"] = int((o["n_resto"] > 0).sum())
    parity["restored_sets_equal"] = bool(np.array_equal(o["n_resto"] > 0, resto[:n_par] > 0))
    # converged: checked problems count when in parity; problems outside the checked sample (only with --parity sample) count by status
    conv_local = int(ok.sum()) + int((status[n_par:] == 0).sum())
    conv_nores_local = int((ok & (resto[:n_par] == 0)).sum()) + int(((status[n_par:] == 0) & (resto[n_par:] == 0)).sum())
    conv_total, conv_nores_total, optimal_total, iters_total, resto_total, checked_total, inpar_total = allsum(
        [conv_local, conv_nores_local, optimal_local, int(iters.sum()), int((resto > 0).sum()), n_par, int(ok.sum())])
    value = conv_total * args.steps / (total_ms * 1e-3)

    # ---- end to end through the C ABI with pinned host buffers (H2D + kernel + D2H timed; at N > 1 the all-gather too)
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
    h_state, h_ref, h_uprev, h_vdes = pin(b["state"]), pin(b["ref"]), pin(b["u_prev"]), pin(b["v_des"])
    solver.set_stream(None)  # back to the handle's own stream
    gather_bytes = 0

    def e2e_step():
        r = solver.solve_batch_records(h_state, h_ref, h_uprev, v_des=h_vdes)
        if world > 1:   # every rank ends the step holding every problem's record, on the host
            d_rec.copy_(torch.from_numpy(r))
            dist.all_gather_into_tensor(d_all, d_rec)
            return d_all.cpu().numpy()
        return r
    for _ in range(2):
        e2e_step()
    barrier()
    w0 = time.perf_counter()
    h2d = d2h = 0
    for _ in range(args.steps):
        e2e_step()
        st = solver.stats()
        h2d, d2h = st["h2d_bytes"], st["d2h_bytes"]
    torch.cuda.synchronize()
    e2e_value = conv_total * args.steps / allmax(time.perf_counter() - w0)
    if world > 1:
        h2d += B * 32; d2h += world * B * 32; gather_bytes = world * B * 32

    # ---- the same with the waypoints generated on the device (mpcb200_solve_batch_on_path): the host sends the
    # state, the path id and the previous command only (60 B/problem instead of 560)
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    for i, pth in enumerate((1, 2, 3)):
        solver.set_path(i, GPSRefTrajectory(mat_filename=pth, traj_horizon=N, traj_dt=0.2).trajectory)
    h_pathof = torch.from_numpy((b["path"] - 1).astype(np.int32)).pin_memory().numpy()
    for _ in range(2):
        solver.solve_batch_on_path(h_state, h_pathof, h_uprev, v_des=h_vdes)
    barrier()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        r2 = solver.solve_batch_on_path(h_state, h_pathof, h_uprev, v_des=h_vdes)
        st2 = solver.stats()
    torch.cuda.synchronize()
    t_op = allmax(time.perf_counter() - w0)
    same_as_ref = bool(np.array_equal(r2["u0"], u0) and np.array_equal(r2["status"], status))
    e2e_on_path = {"value": allsum([float((r2["status"] == 0).sum())])[0] * args.steps / t_op, "unit": "solves/s",
                   "h2d_bytes_per_step": int(st2["h2d_bytes"]), "d2h_bytes_per_step": int(st2["d2h_bytes"]),
                   "bitwise_equal_to_host_references": same_as_ref,
                   "what": "mpcb200_solve_batch_on_path: reference waypoints generated on the device"}

    extras = {}

    def extra(name, fn):
        """the configs beside the headline: outside its timed region, never allowed to break the line"""
        try:
            extras[name] = fn()
        except Exception as ex:
            extras[name] = {"error": repr(ex)}

    def timed_device_solve(Nh, Bh, start_mode, max_iter=None, reps=2, b0=0, rollout_warm=False, min_batch=None, bb=None):
        """min_batch: None = the library's default rule for the kernel layout, 0 = one warp per problem, 1 = one thread per problem"""
        bb = workload.make_batch(Bh, Nh, b0=b0) if bb is None else bb
        kw = {} if max_iter is None else {"max_iter": max_iter}
        sv = capi.Solver(Nh, device=local, start_mode=start_mode, **kw)
        if min_batch is not None:
            sv.set_large_batch_path(min_batch)
        sv.set_stream(stream.cuda_stream)
        dd = {k_: torch.from_numpy(bb[k_]).to(dev) for k_ in ("state", "ref", "u_prev", "v_des")}
        rec = torch.empty((Bh, 4), dtype=torch.float64, device=dev)
        best = 1e30
        for _ in range(1 + reps):
            flush.zero_()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            sv.solve_batch_records_device(Bh, dd["state"], dd["ref"], dd["u_prev"], rec, v_des=dd["v_des"])
            a1.record(stream); torch.cuda.synchronize()
            best = min(best, a0.elapsed_time(a1))
        uu, cc, ss, ii, rr = sharding.unpack_records_np(rec.cpu().numpy())
        sv.close()
        return bb, best, uu.copy(), cc.copy(), ss, ii, rr

    # configs[1]: 4,096 cold solves at N = 8 along path 1 (one GPU's worth: every rank runs the same batch, rank 0 reports)
    def config1():
        bb, ms, uu, cc, ss, ii, rr = timed_device_solve(8, 4096, capi.START_ZERO)
        bb = workload.make_batch(4096, 8, path_ids=(1,))
        sv = capi.Solver(8, device=local); sv.set_stream(stream.cuda_stream)
        dd = {k_: torch.from_numpy(bb[k_]).to(dev) for k_ in ("state", "ref", "u_prev", "v_des")}
        rec = torch.empty((4096, 4), dtype=torch.float64, device=dev)
        ms = 1e30
        for _ in range(4):
            flush.zero_()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            sv.solve_batch_records_device(4096, dd["state"], dd["ref"], dd["u_prev"], rec, v_des=dd["v_des"])
            a1.record(stream); torch.cuda.synchronize()
            ms = min(ms, a0.elapsed_time(a1))
        uu, cc, ss, ii, rr = sharding.unpack_records_np(rec.cpu().numpy())
        tq = time.perf_counter()
        oo = O.solve_batch(O.default_cfg(8, max_iter=int(sv.cfg.max_iter)), bb["state"], bb["ref"], bb["v_des"], bb["u_prev"], n_threads=threads)
        cdt = time.perf_counter() - tq
        sv.close()
        okk, par = parity_counts(uu.copy(), cc.copy(), ss, oo)
        return {"what": "configs[1]: 4,096 cold solves from perturbed states along path1, N=8, one GPU", "kernel_ms": ms,
                "value": float(okk.sum()) / (ms * 1e-3), "unit": "converged solves/s", "mean_iters": float(ii.mean()),
                "restored": int((rr > 0).sum()), "parity_vs_oracle": par,
                "cpu_oracle": {"value": float((oo["status"] == 0).sum()) / cdt, "unit": "solves/s", "cores": threads, "kind": "port"}}

    # configs[3]: 16,384 vehicles x 500 control steps, closed loop on the device, the fleet sharded over the ranks
    def rollout_config3():
        from mkz_mpc_path_follower_b200 import closed_loop
        V, T = args.rollout_vehicles, args.rollout_steps
        trajs = [GPSRefTrajectory(mat_filename=p_) for p_ in (1, 2, 3)]
        rng = np.random.Generator(np.random.Philox(key=20261018))
        nz = rng.normal(size=(V, 3)) * np.array([0.3, 0.3, 0.05])
        path_of = (np.arange(V) % 3).astype(np.int32)
        pose0 = np.stack([trajs[p_].trajectory[0, [4, 5, 3]] for p_ in path_of]) + nz
        lo, hi = sharding.shard_range(V, world, rank)
        sv = capi.Solver(8, device=local)
        for i_, g_ in enumerate(trajs):
            sv.set_path(i_, g_.trajectory)
        sv.rollout(pose0[lo:lo + 64], path_of[lo:lo + 64], 5)    # warm-up (module-load solve, clocks)
        walls = []
        for _ in range(2):     # the first call also allocates the fleet's device buffers and touches the log's pages for the first time
            barrier()
            tq = time.perf_counter()
            out = sv.rollout(pose0[lo:hi], path_of[lo:hi], T)
            walls.append(allmax(time.perf_counter() - tq))
        wall = min(walls)
        kms = allmax(sv.stats()["kernel_ms"])
        launches = sv.stats()["kernel_launches"]
        fused = None
        if launches > 1 and rank == 0 and world == 1:
            # the library ran the per-period pipeline (plant / waypoints / thread-per-problem solve): the fused kernel beside it
            sv.set_large_batch_path(0)
            tq2 = time.perf_counter()
            out_f = sv.rollout(pose0[lo:hi], path_of[lo:hi], T)
            fused = {"wall_s": time.perf_counter() - tq2, "kernel_ms": sv.stats()["kernel_ms"], "kernel": "mpc_rollout_kernel",
                     "statuses_equal": bool(np.array_equal(out_f["log"][:, :, 6], out["log"][:, :, 6])),
                     "max_abs_diff_driving_vehicles": float(np.abs(out_f["log"][:, :, 0:6] - out["log"][:, :, 0:6])[:, (out["log"][:, :, 6] != -1).all(axis=0), :].max())}
            sv.set_large_batch_path(-1)
        log = out["log"]
        solved = log[:, :, 6] >= 0
        err = np.zeros(hi - lo)
        for p_ in range(3):
            m = path_of[lo:hi] == p_
            if m.any():
                err[m] = closed_loop.path_errors(log[-1:, m, :], trajs[p_].trajectory)[0]
        n_solved, n_opt, n_it = allsum([float(solved.sum()), float((log[:, :, 6] == 0).sum()), float(log[:, :, 7].sum())])
        if world > 1:
            ea = torch.zeros(V, dtype=torch.float64, device=dev); ea[lo:hi] = torch.from_numpy(err).to(dev)
            dist.all_reduce(ea, op=dist.ReduceOp.SUM); err = ea.cpu().numpy()
        sv.close()
        return {"what": "configs[3]: %d vehicles x %d control steps (N=8, paths 1-3, warm-started solve each step) through "
                        "mpcb200_rollout, fleet sharded over %d GPU(s)" % (V, T, world), "scaling": "strong",
                "kernels": ("rollout_plant_kernel + rollout_waypoints_kernel + rollout_solve_tpp_kernel per control period" if launches > 1
                            else "mpc_rollout_kernel (one persistent launch)"), "kernel_launches": int(launches), "fused_kernel_for_comparison": fused,
                "wall_s": wall, "wall_s_first_call": walls[0], "kernel_ms": kms, "solves": n_solved, "solves_per_s": n_solved / wall,
                "vehicle_steps_per_s": V * T / wall, "optimal_frac": n_opt / max(1.0, n_solved), "mean_iters": n_it / max(1.0, n_solved),
                "final_path_error_m": {"median": float(np.median(err)), "p99": float(np.quantile(err, 0.99))}}

    # configs[4]: horizon sweep N = 8 / 40 / 80 (N = 20 is the headline), per GPU, from the reference's all-zero start
    # (with its converged fraction inside the iteration cap) and from MPCB200_START_ROLLOUT (opt-in)
    def horizon_sweep():
        res = {}
        Bh = args.sweep_batch     # configs[4]: 1 M problems over 8 GPUs = 131,072 per GPU, at every horizon
        for Nh in (8, 40, 80):
            row = {"batch_per_gpu": Bh}
            bb = workload.make_batch(Bh, Nh, b0=rank * Bh)
            for nm, mode in (("zero_start", capi.START_ZERO), ("rollout_start", capi.START_ROLLOUT)):
                _, ms, uu, cc, ss, ii, rr = timed_device_solve(Nh, Bh, mode, reps=1, bb=bb)
                conv, nit = allsum([float((ss == 0).sum()), float(ii.sum())])
                msx = allmax(ms)
                tpp = Nh <= 10 and Bh >= (16384 if mode == capi.START_ROLLOUT else 32768)     # the library's default rule
                row[nm] = {"kernel": "mpc_solve_tpp_kernel" if tpp else ("mpc_solve_kernel" if Nh <= 31 else "mpc_solve_long_kernel"),
                           "kernel_ms": msx, "converged_frac": conv / (world * Bh), "mean_iters": nit / (world * Bh),
                           "value": conv / (msx * 1e-3), "unit": "converged solves/s", "max_iter": 200,
                           "fp64_tflops": nit * (F_RIC + F_EVAL) * Nh / (msx * 1e-3) / 1e12}
            res["N%d" % Nh] = row
            del bb
        res["what"] = ("configs[4] per GPU (weak; 131,072 per GPU = 1 M problems on 8 GPUs): all-zero start = the reference's start=0.0, "
                       "converged fraction inside the library's 200-iteration cap (under Ipopt's own cap of 3000 every problem converges at "
                       "N = 40 and N = 80: tools/long_horizon_cap.py, DESIGN 5); rollout start = MPCB200_START_ROLLOUT (opt-in, not a "
                       "reference behaviour)")
        return res

    # the two device layouts of the solver on large batches at the reference's own horizon (N = 8): one warp per problem
    # (iterate on chip) against one thread per problem (iterate streamed from HBM, csrc/tpp_solver.cuh); rank 0's GPU only
    def layouts_n8():
        res = {"what": "N = 8, all-zero start, kernel time of ONE launch per layout on the same batch; the default rule "
                       "(mpcb200_set_large_batch_path) picks one thread per problem from 32,768 problems at N <= 10"}
        for Bh in (65536, 262144):
            bb = workload.make_batch(Bh, 8)
            row = {}
            out = {}
            for nm, mb in (("warp_per_problem", 0), ("thread_per_problem", 1)):
                _, ms, uu, cc, ss, ii, rr = timed_device_solve(8, Bh, capi.START_ZERO, reps=1, min_batch=mb, bb=bb)
                out[nm] = (uu, ss, ii)
                row[nm] = {"kernel_ms": ms, "value": float((ss == 0).sum()) / (ms * 1e-3), "unit": "converged solves/s",
                           "converged_frac": float((ss == 0).mean()), "mean_iters": float(ii.mean())}
            (uw, sw_, iw), (ut, st_, it_) = out["warp_per_problem"], out["thread_per_problem"]
            both = (sw_ == 0) & (st_ == 0)
            row["agreement"] = {"status_equal": int((sw_ == st_).sum()), "iters_equal": int((iw == it_).sum()), "of": Bh,
                                "du_gt_1e-5": int((np.abs(uw - ut)[both].max(axis=1) > 1e-5).sum())}
            row["speedup"] = row["warp_per_problem"]["kernel_ms"] / row["thread_per_problem"]["kernel_ms"]
            res["B%d" % Bh] = row
        return res

    # strong scaling of configs[2]: ONE 65,536-problem batch cut into contiguous slices over the ranks
    def strong_64k():
        lo, hi = sharding.shard_range(B, world, rank)
        n = hi - lo
        if world == 1:
            return {"what": "one 65,536 batch on one GPU = the headline", "ms": total_ms / args.steps, "efficiency_vs_one_gpu": 1.0}
        bb = workload.make_batch(n, N, b0=lo)
        dd = {k_: torch.from_numpy(bb[k_]).to(dev) for k_ in ("state", "ref", "u_prev", "v_des")}
        rec = torch.empty((n, 4), dtype=torch.float64, device=dev)
        sizes = [sharding.shard_range(B, world, q)[1] - sharding.shard_range(B, world, q)[0] for q in range(world)]
        solver.set_stream(stream.cuda_stream)
        ms = []
        for i_ in range(2 + args.steps):
            flush.zero_()
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            solver.solve_batch_records_device(n, dd["state"], dd["ref"], dd["u_prev"], rec, v_des=dd["v_des"])
            allrec = sharding.all_gather_records(rec, sizes)
            a1.record(stream); torch.cuda.synchronize()
            if i_ >= 2:
                ms.append(allmax(a0.elapsed_time(a1)))
        solver.set_stream(None)
        st_all = sharding.unpack_records_np(allrec.cpu().numpy())[2]
        one = float(np.mean(kernel_ms_per_rank))     # one GPU's time for 65,536 problems (this run, weak-scaling step)
        m = float(np.mean(ms))
        return {"what": "ONE 65,536-problem batch of configs[2] split over %d GPUs (contiguous slices, all-gather of the records)" % world,
                "ms": m, "value": float((st_all == 0).sum()) / (m * 1e-3), "unit": "Optimal solves/s",
                "efficiency_vs_one_gpu": one / (world * m), "problems_per_gpu": n}

    if not args.no_extras:
        extra("config1", config1)
        extra("rollout_config3", rollout_config3)
        extra("horizon_sweep", horizon_sweep)
        extra("strong_64k", strong_64k)
        if rank == 0:
            extra("layouts_n8", layouts_n8)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant (only) kernel: FP64 CUDA-core pipe, SURVEY 8(d)
    fp64_peak = solver.fp64_peak_tflops()
    k_ms = float(np.mean(kern_ms))
    flops = float(iters.sum()) * (F_RIC + F_EVAL) * N
    achieved = flops / (k_ms * 1e-3) / 1e12
    io_bytes = B * ((4 + 2 + 3 * (N + 1) + 1) * 8 + 3 * 8 + 2 * 4)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    traffic = None
    tr_file = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(tr_file) and N == 20 and B == 65536:   # the capture is of this configuration
        try:
            traffic = json.load(open(tr_file)).get("bytes_per_launch")
        except Exception:
            pass
    roofline = {
        "bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
        "traffic": traffic,
        "peak_source": "FP64 FMA micro-benchmark run in this process (MEASURED_PEAKS.json has no FP64 entry)",
        "flops_model": "sum_p iters_p * (1235 + 310) * N, SURVEY.md 8(d)",
        "kernel": "mpc_solve_kernel", "kernel_ms": k_ms, "kernel_ms_per_rank": kernel_ms_per_rank,
        "hbm": {"achieved": io_bytes / (k_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": io_bytes / (k_ms * 1e-3) / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback of B200_PROFILING.md",
                "algorithmic_bytes_per_solve": io_bytes // B},
    }

    line = {
        "metric": "converged MPC solves/sec at batch 64K, N=20" if (N == 20 and B == 65536) else "converged MPC solves/sec at batch %d per GPU, N=%d" % (B, N),
        "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[%d]: %d solves per GPU from the %s, N=%d, paths 1-3 round-robin, "
                               "perturbed states (SURVEY 8d)" % (2 if (N == 20 and args.start == "zero") else 4, B,
                                                                 "all-zero start (start=0.0)" if args.start == "zero" else "rollout start (opt-in)", N),
                   "batch_per_gpu": B, "horizon": N, "l2": "256 MiB flush between steps (inputs 36 MB < L2)",
                   "start": args.start, "max_iter": int(solver.cfg.max_iter)},
        "converged": {"definition": "status Optimal AND in parity with the oracle on the same inputs (SURVEY 8d), every problem of "
                                    "every rank's slice checked" if args.parity == "full" else "status Optimal; oracle parity on a sample only",
                      "converged_frac": conv_total / (world * B), "optimal_frac": optimal_total / (world * B),
                      "checked": int(checked_total), "in_parity": int(inpar_total)},
        "converged_frac": conv_total / (world * B), "mean_iters": iters_total / (world * B),
        "restored": {"what": "problems whose line search failed where Ipopt would enter its restoration phase (not restated: "
                             "restoration by rollout instead, DESIGN 5); what Ipopt returns on them is unknown",
                     "count": int(resto_total), "frac": resto_total / (world * B),
                     "value_excluding_restored": conv_nores_total * args.steps / (total_ms * 1e-3)},
        "roofline": roofline,
        "cpu_baseline": {"value": float((o["status"] == 0).sum()) / cpu_dt, "unit": "solves/s", "cores": threads, "kind": "port",
                         "seconds": cpu_dt,
                         "sample": "%s %d problems of rank 0's batch, restated CPU interior point (oracle), NOT Ipopt" %
                                   ("all" if n_par == B else "first", n_par)},
        "parity_vs_oracle": parity,
        "ipopt_probe": ipopt_probe(),
        "e2e": {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "gather_bytes_per_step": int(gather_bytes),
                "what": "mpcb200_solve_batch_records with pinned HOST buffers (H2D + kernel + D2H inside the call)" +
                        ("; then the all-gather of the records and its read-back, all inside the timed region" if world > 1 else "")},
        "e2e_on_path": e2e_on_path,
        "gpu_launches": int(args.steps * 1),
        "clocks": clocks,
    }
    line.update(extras)

    if N <= 31:
        # the Frenet-frame variant (MKZMPCPathFollowerFrenet.jl, SURVEY 8 f-3) on the same batch size and horizon, outside the
        # timed region of the headline metric: device-resident inputs, CUDA events on the shared stream, oracle on a sample
        try:
            fb = workload.make_frenet_batch(B, N, b0=rank * B)
            fs = capi.FrenetSolver(N, device=local)
            fs.set_stream(stream.cuda_stream)
            fd = {k_: torch.from_numpy(fb[k_]).to(dev) for k_ in ("state", "kpoly", "u_prev", "v_des")}
            f_u0 = torch.empty((B, 2), dtype=torch.float64, device=dev); f_st = torch.empty(B, dtype=torch.int32, device=dev)
            f_it = torch.empty(B, dtype=torch.int32, device=dev)
            f_u0w = torch.empty_like(f_u0); f_stw = torch.empty_like(f_st); f_itw = torch.empty_like(f_it)
            f_ms = []
            for i in range(3 + args.steps):
                flush.fill_(1)
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fs.solve_batch_device(B, fd["state"], fd["kpoly"], fd["u_prev"], f_u0, v_des=fd["v_des"], status=f_st, iters=f_it)
                e1.record(stream); torch.cuda.synchronize()
                if i >= 3:
                    f_ms.append(e0.elapsed_time(e1))
            fst = f_st.cpu().numpy(); fit = f_it.cpu().numpy()
            # the same batch through the warp-per-problem kernel (the library's default rule takes the thread-per-problem layout
            # for Frenet batches of >= 32,768 problems, >= 16,384 at N <= 10)
            f_tpp = B >= (16384 if N <= 10 else 32768)
            f_warp_ms = None
            if f_tpp:
                fs.set_large_batch_path(0)
                w_ms = []
                for i in range(2):
                    flush.fill_(1)
                    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    fs.solve_batch_device(B, fd["state"], fd["kpoly"], fd["u_prev"], f_u0w, v_des=fd["v_des"], status=f_stw, iters=f_itw)
                    e1.record(stream); torch.cuda.synchronize()
                    w_ms.append(e0.elapsed_time(e1))
                f_warp_ms = float(min(w_ms))
                fs.set_large_batch_path(-1)
            from oracle import oracle as O
            n_s = min(B, 512)
            fo = O.solve_batch_frenet(O.default_cfg_frenet(N, max_iter=int(fs.cfg.max_iter)), fb["state"][:n_s], fb["kpoly"][:n_s],
                                      fb["v_des"][:n_s], fb["u_prev"][:n_s], n_threads=cores)
            fok = (fo["status"] == 0) & (fst[:n_s] == 0)
            line["frenet_variant"] = {
                "value": float((fst == 0).sum()) / (float(np.mean(f_ms)) * 1e-3), "unit": "solves/s",
                "kernel": "mpc_solve_tpp_kernel<1> (thread per problem)" if f_tpp else "mpc_solve_frenet_kernel",
                "warp_per_problem_kernel_ms": f_warp_ms,
                "layouts_agree": None if f_warp_ms is None else {"status_equal": bool((f_stw.cpu().numpy() == fst).all()), "iters_equal": bool((f_itw.cpu().numpy() == fit).all()),
                                                                 "max_abs_du": float(np.abs(f_u0w.cpu().numpy() - f_u0.cpu().numpy()).max())},
                "kernel_ms": float(np.mean(f_ms)), "converged_frac": float((fst == 0).mean()), "mean_iters": float(fit.mean()),
                "fp64_tflops": float(fit.astype(np.float64).sum()) * (F_RIC + F_EVAL) * N / (float(np.mean(f_ms)) * 1e-3) / 1e12,
                "parity_vs_oracle": {"sample": n_s, "status_equal": bool((fo["status"] == fst[:n_s]).all()),
                                     "max_abs_du": float(np.abs(f_u0.cpu().numpy()[:n_s] - fo["u0"])[fok].max())},
                "roofline": frenet_roofline(float(np.mean(f_ms)), B, N) if f_tpp else None,
                "what": "same batch size and horizon, rank 0's slice, all-zero start, workload.make_frenet_batch"}
        except Exception as ex:   # the headline line must not depend on the variant
            line["frenet_variant"] = {"error": repr(ex)}

    if not args.no_latency:
        # single-solve latency through the C ABI (host buffers, H2D + kernel + D2H), warm-started like the
        # control loop; CPU oracle beside it
        from oracle import oracle as O
        s1 = capi.Solver(N, device=local)
        ocfg = O.default_cfg(N)
        nl = 264
        sol = s1.solve_batch(b["state"][:64], b["ref"][:64], b["u_prev"][:64], v_des=b["v_des"][:64], want_traj=True)["traj"]
        lat = {"g_warm": [], "c_warm": [], "g_cold": [], "c_cold": []}
        for i in range(nl):
            j = i % 64
            for mode in ("warm", "cold"):
                # warm: from the problem's own previous solution, like the control loop re-solving 0.1 s later; cold: start=0.0
                wg = sol[j:j + 1].copy() if mode == "warm" else None
                wc = sol[j].copy() if mode == "warm" else None
                a = time.perf_counter()
                s1.solve_batch(b["state"][j:j + 1], b["ref"][j:j + 1], b["u_prev"][j:j + 1], v_des=b["v_des"][j:j + 1], warm=wg)
                lat["g_" + mode].append(time.perf_counter() - a)
                if i < 96:   # the CPU leg is slow from the cold start: a bounded sample
                    a = time.perf_counter()
                    O.solve(ocfg, b["state"][j], b["ref"][j], 1.0, b["u_prev"][j], warm=wc)
                    lat["c_" + mode].append(time.perf_counter() - a)
        pct = lambda v, q: 1e3 * float(np.percentile(v[8:], q))
        line["latency"] = {"gpu_p50_ms": pct(lat["g_warm"], 50), "gpu_p99_ms": pct(lat["g_warm"], 99),
                           "cpu_oracle_p50_ms": pct(lat["c_warm"], 50),
                           "gpu_cold_p50_ms": pct(lat["g_cold"], 50), "gpu_cold_p99_ms": pct(lat["g_cold"], 99),
                           "cpu_oracle_cold_p50_ms": pct(lat["c_cold"], 50),
                           "what": "batch of 1 through the C ABI incl. H2D/D2H (one mpcb200_solve_batch call per solve); warm = start from "
                                   "the problem's previous solution like the control loop, cold = the all-zero start; the oracle is the "
                                   "restated CPU interior point on one thread, NOT Ipopt; closed-loop percentiles: tools/closed_loop_latency.py"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
