#!/usr/bin/env python
"""A/B of the solve kernel's queue order (DESIGN §6, item 3): kernel time of cold-start batches at N = 20 through two builds of
libmpc_b200.so, alternated run by run, each run a process of its own (MPCB200_LIB selects the build).

    python tools/queue_order_ab.py --lib A=path/to/a.so --lib B=path/to/b.so --runs 5 [--batches 2048,8192,65536] [--profile B]

Per run and batch: one warm-up launch, then the best of three launches timed with CUDA events on the handle's stream, a
256 MiB L2 flush before each (what bench.py does).  Every run also returns the records of each batch; the summary says whether
the builds agree bit for bit.  --profile NAME: one more run of that build under torch.profiler, with the device time of each
kernel of the 65,536-problem launch (the queue-key kernel and the sort on their own).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child(batches, out, profile):
    sys.path.insert(0, ROOT)
    import torch
    from mkz_mpc_path_follower_b200 import capi, workload
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    N = 20
    res = {"gpu": torch.cuda.get_device_name(0), "ms": {}}
    recs = {}
    for B in batches:
        b = workload.make_batch(B, N)
        sv = capi.Solver(N)
        sv.set_stream(stream.cuda_stream)
        d = {k: torch.from_numpy(b[k]).to(dev) for k in ("state", "ref", "u_prev", "v_des")}
        rec = torch.empty((B, 4), dtype=torch.float64, device=dev)
        call = lambda: sv.solve_batch_records_device(B, d["state"], d["ref"], d["u_prev"], rec, v_des=d["v_des"])
        call()
        if profile:
            import warnings
            from torch.profiler import ProfilerActivity, profile as prof
            warnings.filterwarnings("ignore", message=".*Profiler clears events")   # one profiled call: nothing is lost
            torch.cuda.synchronize()
            with prof(activities=[ProfilerActivity.CUDA]) as p:
                call()
                torch.cuda.synchronize()
            ev = {}
            for e in p.events():
                if e.device_type.name == "CUDA":
                    ev[e.name[:80]] = ev.get(e.name[:80], 0.0) + e.device_time / 1e3
            res.setdefault("kernels_ms", {})[str(B)] = ev
        best = 1e30
        for _ in range(3):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            call()
            e1.record(stream)
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        res["ms"][str(B)] = best
        res["launches_" + str(B)] = sv.stats()["kernel_launches"]
        recs[str(B)] = rec.cpu().numpy()
        sv.close()
    np.savez(out + ".npz", **recs)
    with open(out + ".json", "w") as f:
        json.dump(res, f)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", required=True, help="NAME=path of a libmpc_b200.so build")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--batches", default="2048,3552,8192,65536")
    ap.add_argument("--profile", default=None)
    ap.add_argument("--child", default=None)
    args = ap.parse_args()
    batches = [int(x) for x in args.batches.split(",")]
    if args.child:
        return child(batches, args.child, args.profile == "yes")
    libs = dict(x.split("=", 1) for x in args.lib)
    tmp = tempfile.mkdtemp()
    runs = {n: [] for n in libs}
    recs = {}

    def run(name, path, tag, profile=False):
        out = os.path.join(tmp, tag)
        env = dict(os.environ, MPCB200_LIB=os.path.abspath(path))
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--lib", "x=y", "--batches", args.batches, "--child", out,
                               "--profile", "yes" if profile else "no"], env=env)
        return json.load(open(out + ".json")), dict(np.load(out + ".npz"))

    for r in range(args.runs):
        for name, path in libs.items():
            res, rc = run(name, path, "%s_%d" % (name, r))
            runs[name].append(res)
            recs.setdefault(name, rc)
            print(json.dumps({"run": r, "build": name, **res}), flush=True)
    names = list(libs)
    summary = {"gpu": runs[names[0]][0]["gpu"], "runs": args.runs, "median_ms": {}, "spread": {}}
    for n in names:
        for B in batches:
            v = np.array([x["ms"][str(B)] for x in runs[n]])
            summary["median_ms"].setdefault(str(B), {})[n] = round(float(np.median(v)), 4)
            summary["spread"].setdefault(str(B), {})[n] = round(float((v.max() - v.min()) / np.median(v)), 4)
    for B in batches:
        m = summary["median_ms"][str(B)]
        summary["median_ms"][str(B)]["%s/%s" % (names[-1], names[0])] = round(m[names[-1]] / m[names[0]], 4)
    summary["bit_identical"] = {str(B): all(np.array_equal(recs[names[0]][str(B)], recs[n][str(B)]) for n in names) for B in batches}
    if args.profile:
        res, _ = run(args.profile, libs[args.profile], "profile", profile=True)
        summary["kernels_ms_" + args.profile] = res.get("kernels_ms")
    print(json.dumps({"summary": summary}))


if __name__ == "__main__":
    main()
