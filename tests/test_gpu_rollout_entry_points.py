"""GPU tests of the three closed-loop entry points, mpcb200_rollout, mpcb200_rollout_w and mpcb200_rollout_frenet, which share
one driver: a Frenet fleet runs on devices[0] of a multi-GPU handle and equals a one-device handle's rollout bit for bit, and
every rejected argument returns MPCB200_EINVAL with a message that names the entry point it came through."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EINVAL = -1


@pytest.fixture(scope="module")
def capi():
    from mkz_mpc_path_follower_b200 import capi as c
    c.lib()
    return c


@pytest.fixture(scope="module")
def trajs():
    from mkz_mpc_path_follower_b200.gps_ref_traj import GPSRefTrajectory
    return [GPSRefTrajectory(mat_filename=p).trajectory for p in (1, 2, 3)]


def fleet(trajs, B, seed):
    """B vehicles near paths 0-2, a few decimetres off with a small heading error"""
    rng = np.random.default_rng(seed)
    path_of = (np.arange(B) % 3).astype(np.int32)
    pose0 = np.stack([trajs[p][(53 * (i + 1)) % (trajs[p].shape[0] - 1500), [4, 5, 3]] + rng.normal(scale=[0.3, 0.3, 0.03])
                      for i, p in enumerate(path_of)])
    return pose0, path_of


def test_frenet_fleet_stays_on_first_device(capi, trajs):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    N, B, T = 8, 64, 30
    pose0, path_of = fleet(trajs, B, seed=5)
    out = {}
    for name, devices in (("one", [0]), ("multi", [0, 1])):
        s = capi.FrenetSolver(N, devices=devices)
        for i, tb in enumerate(trajs):
            s.set_path(i, tb)
        out[name] = s.rollout(pose0, path_of, T)
        out[name + "_launches"] = s.stats()["kernel_launches"]
    assert out["multi_launches"] == 1 and out["one_launches"] == 1   # the fused kernel, on one device
    assert np.array_equal(out["one"]["log"], out["multi"]["log"])
    assert np.array_equal(out["one"]["final_state"], out["multi"]["final_state"])


def _handle(capi, trajs, frenet, N):
    s = capi.FrenetSolver(N) if frenet else capi.Solver(N)
    s.set_path(0, trajs[0])
    return s


def _call(capi, entry, s, B, T, pose0, path_of, window=40.0, w=None):
    L = capi.lib()
    dp = C.POINTER(C.c_double)
    pose = None if pose0 is None else pose0.ctypes.data_as(dp)
    pid = path_of.ctypes.data_as(C.POINTER(C.c_int32))
    log, final = np.empty((max(T, 1), max(B, 1), 8)), np.empty((max(B, 1), 8))
    outs = (log.ctypes.data_as(dp), final.ctypes.data_as(dp))
    if entry == "mpcb200_rollout":
        rc = L.mpcb200_rollout(s._h, B, T, pose, pid, 1, 1.0, *outs)
    elif entry == "mpcb200_rollout_w":
        rc = L.mpcb200_rollout_w(s._h, B, T, pose, pid, 1, 1.0, w.ctypes.data_as(dp), *outs)
    else:
        rc = L.mpcb200_rollout_frenet(s._h, B, T, pose, pid, float(window), 8.0, 1, *outs)
    return rc, L.mpcb200_last_error(s._h).decode()


CASES = {
    "mpcb200_rollout": ["B<0", "T<0", "model", "pose NULL", "path unset"],
    "mpcb200_rollout_w": ["B<0", "T<0", "model", "pose NULL", "path unset", "NaN weight"],
    "mpcb200_rollout_frenet": ["B<0", "T<0", "model", "N>31", "window", "pose NULL", "path unset"],
}


@pytest.mark.parametrize("entry,case", [(e, c) for e, cs in CASES.items() for c in cs])
def test_rejected_arguments_name_the_entry_point(capi, trajs, entry, case):
    frenet = entry == "mpcb200_rollout_frenet"
    N = 40 if case == "N>31" else 8
    s = _handle(capi, trajs, frenet != (case == "model"), N)
    B, T = 4, 3
    pose0 = np.tile(trajs[0][300, [4, 5, 3]], (B, 1))
    path_of = np.zeros(B, dtype=np.int32)
    w = np.tile([9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0], (B, 1))
    window = 40.0
    if case == "B<0":
        B = -1
    elif case == "T<0":
        T = -1
    elif case == "window":
        window = 2.0
    elif case == "pose NULL":
        pose0 = None
    elif case == "path unset":
        path_of[2] = 1
    elif case == "NaN weight":
        w[3, 5] = np.nan
    rc, msg = _call(capi, entry, s, B, T, pose0, path_of, window=window, w=w)
    assert rc == EINVAL, (rc, msg)
    assert msg.startswith(entry + ":"), msg
    if case == "path unset":
        assert "vehicle 2 uses path 1" in msg, msg
    if case == "NaN weight":
        assert "weight 5 of vehicle 3" in msg, msg
    if case == "N>31":
        return   # no Frenet rollout runs at N > 31
    # the handle still serves a valid call (for the model case through the entry point of its own model)
    ok_entry = entry if case != "model" else ("mpcb200_rollout" if frenet else "mpcb200_rollout_frenet")
    rc, msg = _call(capi, ok_entry, s, 4, 3, np.tile(trajs[0][300, [4, 5, 3]], (4, 1)), np.zeros(4, dtype=np.int32),
                    w=np.tile([9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0], (4, 1)))
    assert rc == 0, msg
