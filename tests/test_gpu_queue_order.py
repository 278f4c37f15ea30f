"""Queue order of large cold-start batches (mpc_b200.cu: queue_key_kernel, queue_order, mpc_solve_kernel<PW, 1>): a batch of
more than one wave of resident teams (mpcb200_create says how much more) is solved longest predicted solve first, which must
change nothing but the timing.  The reference is the same problems solved in slices below that size, in counter order."""
import numpy as np
import pytest

from mkz_mpc_path_follower_b200 import workload as W

pytestmark = pytest.mark.gpu

SLICE = 1000     # below one wave of resident teams on any GPU with 84 SMs or more: never ordered


@pytest.fixture(scope="module")
def capi():
    from mkz_mpc_path_follower_b200 import capi as c
    c.lib()
    return c


def _ordered(s, b, B):
    """Whether the handle orders a cold batch of B problems: the key kernel and the sort launch before the solve."""
    s.solve_batch(b["state"][:B], b["ref"][:B], b["u_prev"][:B], v_des=b["v_des"][:B])
    return s.stats()["kernel_launches"] == 3


def _min_ordered_batch(s, b):
    """The smallest batch the handle orders, found by bisection over [SLICE, len(b)] (it depends on the GPU's SM count and the
    kernel's occupancy)."""
    lo, hi = SLICE, len(b["v_des"])
    assert not _ordered(s, b, lo) and _ordered(s, b, hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (lo, mid) if _ordered(s, b, mid) else (mid, hi)
    return hi


@pytest.mark.parametrize("N", [8, 20])
def test_ordered_batch_equals_counter_order(capi, N):
    """Every output of an ordered batch equals, bit for bit, the output of the same problems solved in unordered slices; a size
    that is no multiple of the four teams of a block, and more than the order threshold."""
    B = 8192 + 1237
    b = W.make_batch(B, N, b0=3 * 65536)
    s = capi.Solver(N)
    g = s.solve_batch(b["state"], b["ref"], b["u_prev"], v_des=b["v_des"], want_traj=True)
    assert s.stats()["kernel_launches"] == 3
    ref = {k: [] for k in ("u0", "cost", "status", "iters", "traj")}
    for lo in range(0, B, SLICE):
        hi = min(B, lo + SLICE)
        r = s.solve_batch(b["state"][lo:hi], b["ref"][lo:hi], b["u_prev"][lo:hi], v_des=b["v_des"][lo:hi], want_traj=True)
        assert s.stats()["kernel_launches"] == 1
        for k in ref:
            ref[k].append(r[k])
    for k in ref:
        assert np.array_equal(g[k], np.concatenate(ref[k]), equal_nan=True), k


def test_ordered_batch_writes_every_record_once(capi):
    """Device buffers: the record array starts as NaN, and after an ordered solve every record holds its problem's answer (the
    order is a permutation: a problem solved twice would leave another one unsolved); the threshold itself is ordered, one
    problem less is not."""
    import torch
    from mkz_mpc_path_follower_b200 import sharding
    N = 20
    b = W.make_batch(8192, N, b0=5 * 65536)
    s = capi.Solver(N)
    B0 = _min_ordered_batch(s, b)
    dev = torch.device("cuda", 0)
    d = {k: torch.from_numpy(b[k]).to(dev) for k in ("state", "ref", "u_prev", "v_des")}
    ref = s.solve_batch_records(b["state"][:SLICE], b["ref"][:SLICE], b["u_prev"][:SLICE], v_des=b["v_des"][:SLICE])
    for B, launches in ((B0, 3), (B0 - 1, 1)):
        rec = torch.full((B, 4), float("nan"), dtype=torch.float64, device=dev)
        s.solve_batch_records_device(B, d["state"], d["ref"], d["u_prev"], rec, v_des=d["v_des"])
        torch.cuda.synchronize()
        assert s.stats()["kernel_launches"] == launches
        r = rec.cpu().numpy()
        assert not np.isnan(r).any()
        u0, cost, status, iters, _ = sharding.unpack_records_np(r)
        assert ((status >= 0) & (status <= 4)).all() and (iters >= 0).all()
        assert np.array_equal(r[:SLICE], ref)
