"""bench.py's reference arm runs on the host cores (no GPU): its JSON line must carry the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-sample", "48", "--horizon", "8"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "solves/s" and line["higher_is_better"] is True
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["e2e"]["value"] == line["value"] and line["vs_baseline"] is None and line["dtype"] == "f64"
    assert "workload" in line["config"]


NAMES = ("index", "u0", "cost", "status", "iters", "restorations")


def _load_dump(d):
    out = {k: np.load(os.path.join(d, k + ".npy")) for k in NAMES}
    for k, a in out.items():
        assert a.dtype == np.float64, k
    return out


def test_reference_arm_dump_outputs(tmp_path, oracle):
    """--dump-outputs writes the last timed step's results: with --steps 2 and 48 problems a step, problems 48..95."""
    d = str(tmp_path / "out")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-sample", "48", "--horizon", "8", "--dump-outputs", d], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    g = _load_dump(d)
    assert np.array_equal(g["index"], np.arange(48, 96)) and g["u0"].shape == (48, 2) and g["cost"].shape == (48,)
    from mkz_mpc_path_follower_b200 import workload
    b = workload.make_batch(48, 8, b0=48)
    o = oracle.solve_batch(oracle.default_cfg(8), b["state"], b["ref"], b["v_des"], b["u_prev"], n_threads=2)
    for k in ("u0", "cost", "status", "iters"):
        assert np.array_equal(g[k], o[k].astype(np.float64)), k


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_dump_outputs_sample_is_bounded_and_fixed(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT", 1 << 20)
    n = 100000
    arrays = {"u0": np.arange(2 * n, dtype=np.float64).reshape(n, 2), "status": np.arange(n, dtype=np.int32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), np.arange(n), arrays)
    a, b = ({k: np.load(str(tmp_path / d / (k + ".npy"))) for k in ("index", "u0", "status")} for d in ("a", "b"))
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))) <= 1 << 20
    assert 0 < a["index"].shape[0] < n and np.all(np.diff(a["index"]) > 0)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["u0"], arrays["u0"][a["index"].astype(np.int64)]) and np.array_equal(a["status"], a["index"])


@pytest.mark.gpu
def test_gpu_arm_dump_outputs(tmp_path):
    """The headline path's dump is the record the library returns for the same batch."""
    d = str(tmp_path / "out")
    B, N = 1024, 20
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--batch", str(B),
                          "--horizon", str(N), "--no-extras", "--no-latency", "--parity", "sample", "--cpu-sample", "64",
                          "--dump-outputs", d], capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    g = _load_dump(d)
    assert np.array_equal(g["index"], np.arange(B))
    from mkz_mpc_path_follower_b200 import capi, sharding, workload
    b = workload.make_batch(B, N)
    s = capi.Solver(N)
    u0, cost, status, iters, resto = sharding.unpack_records_np(s.solve_batch_records(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"]))
    for k, v in (("u0", u0), ("cost", cost), ("status", status), ("iters", iters), ("restorations", resto)):
        assert np.array_equal(g[k], v.astype(np.float64)), k
