"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol
include/mpc_b200.h declares (no compute without a GPU), and it refuses to run without one."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "mpc_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mpcb200_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported():
    from mkz_mpc_path_follower_b200 import capi
    L = capi.lib()
    names = _declared()
    assert "mpcb200_solve_batch" in names and "mpcb200_create" in names and len(names) >= 10
    for n in names:
        assert hasattr(L, n), n
    hdr = open(os.path.join(ROOT, "include", "mpc_b200.h")).read()
    assert L.mpcb200_version() == int(re.search(r"#define MPCB200_VERSION (\d+)", hdr).group(1))


def test_default_config_matches_reference_constants():
    from mkz_mpc_path_follower_b200 import capi
    c = capi.default_config(8)
    # MKZMPCPathFollower.jl:28-48
    assert (c.N, c.dt, c.dt_control, c.L_a, c.L_b) == (8, 0.2, 0.1, 1.108, 1.742)
    assert (c.v_min, c.v_max, c.a_max, c.steer_max, c.a_dmax, c.steer_dmax) == (0.0, 20.0, 1.0, 0.5, 1.5, 0.5)
    assert c.tol == 1e-8 and c.start_mode == capi.START_ZERO


BAD_CONSTANTS = [(f, v) for f in ("dt", "dt_control", "L_a", "L_b", "v_min", "v_max", "a_max", "steer_max", "a_dmax", "steer_dmax", "tol")
                 for v in (float("inf"), float("-inf"), float("nan"))] + [("L_a", -0.1), ("L_a", -1e-300)]


@pytest.mark.parametrize("frenet", [False, True], ids=["xy", "frenet"])
@pytest.mark.parametrize("field,value", BAD_CONSTANTS)
def test_create_refuses_bad_constant(field, value, frenet):
    """A constant that is not finite, or a negative L_a, is refused before any device is touched (MPCB200_EINVAL, the message
    names the field): an infinite dt or bound or a NaN L_a would otherwise reach kcfg_finalize, dtLb and rfrac."""
    from mkz_mpc_path_follower_b200 import capi
    with pytest.raises(capi.MpcB200Error) as e:
        (capi.FrenetSolver if frenet else capi.Solver)(8, **{field: value})
    assert e.value.code == -1 and ("model constant %s = " % field) in str(e.value), str(e.value)


def test_create_accepts_edge_constants():
    """L_a = 0 (the rear axle as reference point) and large finite bounds are valid: without a GPU they get as far as the
    device query (MPCB200_ENODEVICE)."""
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    from mkz_mpc_path_follower_b200 import capi
    for kw in (dict(L_a=0.0), dict(v_min=-1e300, v_max=1e300, a_max=1e300, a_dmax=1e300, steer_dmax=1e300, tol=1e300)):
        if has_gpu:
            capi.Solver(8, **kw).close()
            continue
        with pytest.raises(capi.MpcB200Error) as e:
            capi.Solver(8, **kw)
        assert e.value.code == -2, str(e.value)


def test_no_cpu_fallback():
    """Without a CUDA device the product must fail loudly, not fall back."""
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("GPU present")
    from mkz_mpc_path_follower_b200 import capi
    with pytest.raises(capi.MpcB200Error) as e:
        capi.Solver(8)
    assert e.value.code == -2
    # nothing in the package imports the oracle
    pkg = os.path.join(ROOT, "mkz_mpc_path_follower_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            assert "oracle" not in open(os.path.join(pkg, fn)).read().replace("# oracle", ""), fn
