"""ctypes binding of libmpc_b200.so (include/mpc_b200.h).

The library is the product: if it is missing or cannot be loaded this module raises --
there is no CPU or PyTorch fallback anywhere in the package.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MPCB200_LIB") or os.path.join(_HERE, "libmpc_b200.so")

OPTIMAL, INFEASIBLE, UNBOUNDED, USERLIMIT, ERROR = 0, 1, 2, 3, 4
STATUS_SYMBOLS = {0: "Optimal", 1: "Infeasible", 2: "Unbounded", 3: "UserLimit", 4: "Error"}
HOST, DEVICE = 0, 1
START_ZERO, START_ROLLOUT = 0, 1
# the per-vehicle fields of rollout(..., metrics=True) (MPCB200_METRICS, include/mpc_b200.h), in column order
ROLLOUT_METRICS = ("n_solved", "path_err_mean", "path_err_rms", "path_err_max", "heading_err_rms", "heading_err_max",
                   "acc_rate_rms", "steer_rate_rms", "n_not_optimal", "iters_total", "s_last", "stop_period")


class Config(C.Structure):
    _fields_ = [("N", C.c_int32), ("max_iter", C.c_int32), ("start_mode", C.c_int32), ("device", C.c_int32),
                ("dt", C.c_double), ("dt_control", C.c_double), ("L_a", C.c_double), ("L_b", C.c_double),
                ("v_min", C.c_double), ("v_max", C.c_double), ("a_max", C.c_double), ("steer_max", C.c_double),
                ("a_dmax", C.c_double), ("steer_dmax", C.c_double), ("tol", C.c_double),
                ("n_devices", C.c_int32), ("devices", C.c_int32 * 8)]


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("kernel_ms", C.c_float)]


class MpcB200Error(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "libmpc_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libmpc_b200.so is not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "or `make -C mkz_mpc_path_follower_b200/csrc`.  There is no fallback path." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_void_p
    L.mpcb200_version.restype = C.c_int
    L.mpcb200_default_config.argtypes = [C.POINTER(Config), C.c_int32]
    L.mpcb200_create.argtypes = [C.POINTER(vp), C.POINTER(Config)]
    L.mpcb200_destroy.argtypes = [vp]
    L.mpcb200_set_cost.argtypes = [vp, dp]
    L.mpcb200_set_stream.argtypes = [vp, vp]
    L.mpcb200_set_large_batch_path.argtypes = [vp, C.c_int64]
    L.mpcb200_solve_batch.argtypes = [vp, C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int32]
    L.mpcb200_solve_batch_w.argtypes = [vp, C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int32]
    L.mpcb200_solve_batch_records.argtypes = [vp, C.c_int64, vp, vp, vp, vp, vp, vp, vp, C.c_int32]
    L.mpcb200_get_restorations.argtypes = [vp, C.c_int64, vp]
    L.mpcb200_create_frenet.argtypes = [C.POINTER(vp), C.POINTER(Config)]
    L.mpcb200_set_cost_frenet.argtypes = [vp, dp]
    L.mpcb200_solve_batch_frenet.argtypes = [vp, C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int32]
    L.mpcb200_solve_batch_frenet_w.argtypes = [vp, C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int32]
    L.mpcb200_solve_batch_on_path.argtypes = [vp, C.c_int64, vp, vp, C.c_int32, C.c_double, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int32]
    L.mpcb200_solve_batch_frenet_on_path.argtypes = [vp, C.c_int64, vp, vp, C.c_double, C.c_double, C.c_int32] + [vp] * 11 + [C.c_int32]
    L.mpcb200_set_path.argtypes = [vp, C.c_int32, C.c_int32, dp, dp, dp, dp, dp]
    L.mpcb200_rollout.argtypes = [vp, C.c_int64, C.c_int32, dp, ip, C.c_int32, C.c_double, dp, dp]
    L.mpcb200_rollout_w.argtypes = [vp, C.c_int64, C.c_int32, dp, ip, C.c_int32, C.c_double, dp, dp, dp]
    L.mpcb200_rollout_frenet.argtypes = [vp, C.c_int64, C.c_int32, dp, ip, C.c_double, C.c_double, C.c_int32, dp, dp]
    L.mpcb200_rollout_metrics.argtypes = [vp, C.c_int64, C.c_int32, dp, ip, C.c_int32, C.c_double, dp, dp, dp, dp]
    L.mpcb200_rollout_frenet_metrics.argtypes = [vp, C.c_int64, C.c_int32, dp, ip, C.c_double, C.c_double, C.c_int32, dp, dp, dp]
    L.mpcb200_rollout_frenet_w.argtypes = [vp, C.c_int64, C.c_int32, dp, ip, C.c_double, C.c_double, C.c_int32, dp, dp, dp, dp]
    L.mpcb200_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.mpcb200_fp64_peak.argtypes = [vp, dp]
    L.mpcb200_last_error.argtypes = [vp]
    L.mpcb200_last_error.restype = C.c_char_p
    _lib = L
    return L


def default_config(N=8, devices=None, **overrides):
    """devices: list of CUDA ordinals for a multi-GPU handle (mpcb200_config.devices / n_devices); None = `device`."""
    c = Config()
    rc = lib().mpcb200_default_config(C.byref(c), N)
    if rc != 0:
        raise MpcB200Error(rc, "default_config")
    for k, v in overrides.items():
        setattr(c, k, v)
    if devices is not None:
        devices = list(devices)
        if not 1 <= len(devices) <= 8:
            raise ValueError("devices: 1 to 8 CUDA ordinals")
        c.n_devices = len(devices)
        for i, d in enumerate(devices):
            c.devices[i] = int(d)
    return c


def _ptr(a):
    """numpy array -> host pointer; torch CUDA tensor -> device pointer; None -> NULL."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


def _weight_rows(weights, B, n, who):
    """Per-problem cost weights: (B, n) float64 numpy array (host calls)."""
    w = np.ascontiguousarray(weights, dtype=np.float64)
    if w.shape != (B, n):
        raise ValueError("%s: weights must be (B,%d) = (%d,%d), got %s" % (who, n, B, n, w.shape))
    return w


def _weight_rows_device(weights, B, n, who):
    """Per-problem cost weights on the device: a (B, n) tensor, passed as it is (float64, contiguous)."""
    if tuple(weights.shape) != (B, n):
        raise ValueError("%s: weights must be (B,%d) = (%d,%d), got %s" % (who, n, B, n, tuple(weights.shape)))
    return weights


class Solver(object):
    """One handle = one GPU + one stream (mpcb200_create)."""

    def __init__(self, N=8, config=None, **overrides):
        self.cfg = config if config is not None else default_config(N, **overrides)
        self.N = self.cfg.N
        self._h = C.c_void_p()
        rc = self._create()(C.byref(self._h), C.byref(self.cfg))
        if rc != 0:
            raise MpcB200Error(rc, lib().mpcb200_last_error(None).decode())

    def _create(self):
        return lib().mpcb200_create

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().mpcb200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise MpcB200Error(rc, lib().mpcb200_last_error(self._h).decode())

    def set_cost(self, w):
        w = np.ascontiguousarray(w, dtype=np.float64)
        assert w.shape == (8,)
        self._check(lib().mpcb200_set_cost(self._h, w.ctypes.data_as(C.POINTER(C.c_double))))

    def set_large_batch_path(self, min_batch=-1):
        """Batches of at least `min_batch` problems (per device) use the thread-per-problem kernel; 0: never; < 0: default rule."""
        self._check(lib().mpcb200_set_large_batch_path(self._h, int(min_batch)))

    def set_stream(self, cuda_stream_ptr):
        self._check(lib().mpcb200_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def solve_batch(self, state, ref, u_prev, v_des=None, warm=None, want_traj=False, want_aux=True, weights=None):
        """Host (numpy) arrays in, numpy arrays out.  state (B,4); ref (B,3,N+1); u_prev (B,2)
        = (d_f_current, acc_current); v_des (B,) or None; warm (B,6N+4) in/out or None.
        weights (B,8) in update_cost order (cx, cy, cp, cv, cda, cdd, ca, cd), one row per problem (mpcb200_solve_batch_w),
        or None: the handle's weights (set_cost)."""
        N = self.N
        state = np.ascontiguousarray(state, dtype=np.float64)
        B = state.shape[0]
        ref = np.ascontiguousarray(ref, dtype=np.float64)
        u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
        if state.shape != (B, 4) or ref.shape != (B, 3, N + 1) or u_prev.shape != (B, 2):
            raise ValueError("solve_batch: expected state (B,4), ref (B,3,N+1), u_prev (B,2)")
        if v_des is not None:
            v_des = np.ascontiguousarray(v_des, dtype=np.float64)
            if v_des.shape != (B,):
                raise ValueError("solve_batch: v_des must be (B,)")
        if warm is not None:
            if not (isinstance(warm, np.ndarray) and warm.dtype == np.float64 and warm.flags.c_contiguous
                    and warm.shape == (B, 6 * N + 4)):
                raise ValueError("solve_batch: warm must be a C-contiguous float64 (B,6N+4) array (updated in place)")
        u0 = np.empty((B, 2))
        cost = np.empty(B) if want_aux else None
        status = np.empty(B, dtype=np.int32) if want_aux else None
        iters = np.empty(B, dtype=np.int32) if want_aux else None
        traj = np.empty((B, 6 * N + 4)) if want_traj else None
        if weights is None:
            self._check(lib().mpcb200_solve_batch(self._h, B, _ptr(state), _ptr(ref), _ptr(v_des), _ptr(u_prev), _ptr(warm),
                                                  _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj), HOST))
        else:
            w = _weight_rows(weights, B, 8, "solve_batch")
            self._check(lib().mpcb200_solve_batch_w(self._h, B, _ptr(state), _ptr(ref), _ptr(v_des), _ptr(u_prev), _ptr(warm), _ptr(w),
                                                    _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj), HOST))
        return {"u0": u0, "cost": cost, "status": status, "iters": iters, "traj": traj}

    def solve_batch_on_path(self, state, path_of, u_prev, track_using_time=True, target_vel=1.0, v_des=None, warm=None,
                            want_traj=False, want_ref=False):
        """mpcb200_solve_batch_on_path: like solve_batch, but the waypoints are generated on the device from the
        path tables given to set_path (get_waypoints of ref_gps_traj.py).  path_of (B,) in 0..2.  Returns the
        solve_batch dict plus "stop" (B,) and, with want_ref, "ref" (B,3,N+1)."""
        N = self.N
        state = np.ascontiguousarray(state, dtype=np.float64)
        B = state.shape[0]
        path_of = np.ascontiguousarray(path_of, dtype=np.int32)
        u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
        if state.shape != (B, 4) or path_of.shape != (B,) or u_prev.shape != (B, 2):
            raise ValueError("solve_batch_on_path: expected state (B,4), path_of (B,), u_prev (B,2)")
        if v_des is not None:
            v_des = np.ascontiguousarray(v_des, dtype=np.float64)
            if v_des.shape != (B,):
                raise ValueError("solve_batch_on_path: v_des must be (B,)")
        if warm is not None:
            if not (isinstance(warm, np.ndarray) and warm.dtype == np.float64 and warm.flags.c_contiguous
                    and warm.shape == (B, 6 * N + 4)):
                raise ValueError("solve_batch_on_path: warm must be a C-contiguous float64 (B,6N+4) array (updated in place)")
        u0 = np.empty((B, 2)); cost = np.empty(B)
        status = np.empty(B, dtype=np.int32); iters = np.empty(B, dtype=np.int32); stop = np.empty(B, dtype=np.int32)
        traj = np.empty((B, 6 * N + 4)) if want_traj else None
        ref = np.empty((B, 3, N + 1)) if want_ref else None
        self._check(lib().mpcb200_solve_batch_on_path(self._h, B, _ptr(state), _ptr(path_of), int(bool(track_using_time)), float(target_vel),
                                                      _ptr(v_des), _ptr(u_prev), _ptr(warm), _ptr(u0), _ptr(cost), _ptr(status),
                                                      _ptr(iters), _ptr(traj), _ptr(ref), _ptr(stop), HOST))
        return {"u0": u0, "cost": cost, "status": status, "iters": iters, "traj": traj, "ref": ref, "stop": stop}

    def solve_batch_on_path_device(self, B, state, path_of, u_prev, u0, track_using_time=True, target_vel=1.0, v_des=None,
                                   warm=None, cost=None, status=None, iters=None, traj=None, ref_out=None, stop=None):
        """Device pointers (torch CUDA tensors); only enqueues on the handle's stream."""
        self._check(lib().mpcb200_solve_batch_on_path(self._h, B, _ptr(state), _ptr(path_of), int(bool(track_using_time)), float(target_vel),
                                                      _ptr(v_des), _ptr(u_prev), _ptr(warm), _ptr(u0), _ptr(cost), _ptr(status),
                                                      _ptr(iters), _ptr(traj), _ptr(ref_out), _ptr(stop), DEVICE))

    def solve_batch_records(self, state, ref, u_prev, v_des=None, warm=None):
        """mpcb200_solve_batch_records with host arrays: returns the (B,4) float64 array of packed 32-byte records
        (unpack with sharding.unpack_records_np)."""
        N = self.N
        state = np.ascontiguousarray(state, dtype=np.float64)
        B = state.shape[0]
        ref = np.ascontiguousarray(ref, dtype=np.float64); u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
        if state.shape != (B, 4) or ref.shape != (B, 3, N + 1) or u_prev.shape != (B, 2):
            raise ValueError("solve_batch_records: expected state (B,4), ref (B,3,N+1), u_prev (B,2)")
        if v_des is not None:
            v_des = np.ascontiguousarray(v_des, dtype=np.float64)
        rec = np.empty((B, 4))
        self._check(lib().mpcb200_solve_batch_records(self._h, B, _ptr(state), _ptr(ref), _ptr(v_des), _ptr(u_prev), _ptr(warm),
                                                      _ptr(rec), None, HOST))
        return rec

    def solve_batch_records_device(self, B, state, ref, u_prev, rec, v_des=None, warm=None, traj=None):
        """Device pointers; the kernel writes the (B,4) f64 record tensor `rec` itself; only enqueues on the handle's stream."""
        self._check(lib().mpcb200_solve_batch_records(self._h, B, _ptr(state), _ptr(ref), _ptr(v_des), _ptr(u_prev), _ptr(warm),
                                                      _ptr(rec), _ptr(traj), DEVICE))

    def restorations(self, B):
        """Per-problem count of restorations by rollout in the last solve_batch* call (mpcb200_get_restorations)."""
        out = np.empty(B, dtype=np.int32)
        self._check(lib().mpcb200_get_restorations(self._h, B, _ptr(out)))
        return out

    def solve_batch_device(self, B, state, ref, u_prev, u0, v_des=None, warm=None, cost=None, status=None,
                           iters=None, traj=None, weights=None):
        """Device pointers (torch CUDA tensors, float64 / int32, contiguous); only enqueues on the
        handle's stream.  weights: (B,8) float64 tensor, one row per problem (a bad row gives that problem
        status ERROR), or None: the handle's weights."""
        if weights is None:
            self._check(lib().mpcb200_solve_batch(self._h, B, _ptr(state), _ptr(ref), _ptr(v_des), _ptr(u_prev), _ptr(warm),
                                                  _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj), DEVICE))
        else:
            w = _weight_rows_device(weights, B, 8, "solve_batch_device")
            self._check(lib().mpcb200_solve_batch_w(self._h, B, _ptr(state), _ptr(ref), _ptr(v_des), _ptr(u_prev), _ptr(warm), _ptr(w),
                                                    _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj), DEVICE))

    def set_path(self, path_id, traj_table):
        """traj_table: the (n,7) table of GPSRefTrajectory.trajectory (ref_gps_traj.py:106); path_id 0..2."""
        cols = [np.ascontiguousarray(traj_table[:, i], dtype=np.float64) for i in (0, 4, 5, 3, 6)]
        dp = C.POINTER(C.c_double)
        self._check(lib().mpcb200_set_path(self._h, int(path_id), int(traj_table.shape[0]), *[c.ctypes.data_as(dp) for c in cols]))

    def rollout(self, pose0, path_of, T, track_using_time=True, target_vel=1.0, want_log=True, weights=None, metrics=False):
        """Closed-loop Monte-Carlo rollout on the device (mpcb200_rollout).  pose0 (B,3); path_of (B,) in 0..2
        (ids given to set_path).  Returns log (T,B,8) = x,y,psi,v,acc_cmd,df_cmd,status,iters and final (B,8).
        weights (B,8): each vehicle's cost weights for all its control periods (mpcb200_rollout_w), or None: the handle's.
        metrics: also the per-vehicle tracking metrics accumulated on the device (mpcb200_rollout_metrics), out["metrics"] (B,12)
        with the columns of ROLLOUT_METRICS; with want_log=False no log is transferred at all."""
        pose0 = np.ascontiguousarray(np.atleast_2d(pose0), dtype=np.float64)
        B = pose0.shape[0]
        path_of = np.ascontiguousarray(path_of, dtype=np.int32)
        if pose0.shape != (B, 3) or path_of.shape != (B,):
            raise ValueError("rollout: pose0 must be (B,3) and path_of (B,)")
        log = np.empty((T, B, 8)) if want_log else None
        final = np.empty((B, 8))
        dp = C.POINTER(C.c_double)
        args = [pose0.ctypes.data_as(dp), path_of.ctypes.data_as(C.POINTER(C.c_int32)), int(bool(track_using_time)), float(target_vel)]
        outs = [None if log is None else log.ctypes.data_as(dp), final.ctypes.data_as(dp)]
        w = None if weights is None else _weight_rows(weights, B, 8, "rollout")
        if metrics:
            met = np.empty((B, len(ROLLOUT_METRICS)))
            self._check(lib().mpcb200_rollout_metrics(self._h, B, int(T), *args, None if w is None else w.ctypes.data_as(dp), *outs,
                                                      met.ctypes.data_as(dp)))
            return {"log": log, "final_state": final, "metrics": met}
        if w is None:
            self._check(lib().mpcb200_rollout(self._h, B, int(T), *args, *outs))
        else:
            self._check(lib().mpcb200_rollout_w(self._h, B, int(T), *args, w.ctypes.data_as(dp), *outs))
        return {"log": log, "final_state": final}

    def stats(self):
        s = Stats()
        self._check(lib().mpcb200_get_stats(self._h, C.byref(s)))
        return {"kernel_launches": s.kernel_launches, "h2d_bytes": s.h2d_bytes, "d2h_bytes": s.d2h_bytes,
                "kernel_ms": s.kernel_ms}

    def fp64_peak_tflops(self):
        v = C.c_double()
        self._check(lib().mpcb200_fp64_peak(self._h, C.byref(v)))
        return v.value


class FrenetSolver(Solver):
    """Frenet-frame variant (mpcb200_create_frenet; scripts/mpc_utils/MKZMPCPathFollowerFrenet.jl): 3 <= N <= 95."""

    def _create(self):
        return lib().mpcb200_create_frenet

    def set_cost(self, w):
        """update_cost order of MKZMPCPathFollowerFrenet.jl:158-169: cey, cep, cev, cda, cdd, ca, cd."""
        w = np.ascontiguousarray(w, dtype=np.float64)
        assert w.shape == (7,)
        self._check(lib().mpcb200_set_cost_frenet(self._h, w.ctypes.data_as(C.POINTER(C.c_double))))

    def set_large_batch_path(self, min_batch=-1):
        """Batches of at least `min_batch` problems use the thread-per-problem kernel (TppSolverT<1>); 0: never; < 0: the default rule."""
        self._check(lib().mpcb200_set_large_batch_path(self._h, int(min_batch)))

    def solve_batch(self, state, k_coeffs, u_prev, v_des=None, warm=None, want_traj=False, want_aux=True, weights=None):
        """state (B,4) = s, ey, epsi, v; k_coeffs (B,4) highest degree first; u_prev (B,2) = (d_f_current, acc_current);
        warm / traj (B,6N+4) = s, ey, v, epsi, d_f, acc.  weights (B,7) in set_cost's order (cey, cep, cev, cda, cdd, ca, cd),
        one row per problem (mpcb200_solve_batch_frenet_w), or None: the handle's weights."""
        N = self.N
        state = np.ascontiguousarray(state, dtype=np.float64)
        B = state.shape[0]
        k_coeffs = np.ascontiguousarray(k_coeffs, dtype=np.float64)
        u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
        if state.shape != (B, 4) or k_coeffs.shape != (B, 4) or u_prev.shape != (B, 2):
            raise ValueError("solve_batch: expected state (B,4), k_coeffs (B,4), u_prev (B,2)")
        if v_des is not None:
            v_des = np.ascontiguousarray(v_des, dtype=np.float64)
            if v_des.shape != (B,):
                raise ValueError("solve_batch: v_des must be (B,)")
        if warm is not None:
            if not (isinstance(warm, np.ndarray) and warm.dtype == np.float64 and warm.flags.c_contiguous
                    and warm.shape == (B, 6 * N + 4)):
                raise ValueError("solve_batch: warm must be a C-contiguous float64 (B,6N+4) array (updated in place)")
        u0 = np.empty((B, 2))
        cost = np.empty(B) if want_aux else None
        status = np.empty(B, dtype=np.int32) if want_aux else None
        iters = np.empty(B, dtype=np.int32) if want_aux else None
        traj = np.empty((B, 6 * N + 4)) if want_traj else None
        if weights is None:
            self._check(lib().mpcb200_solve_batch_frenet(self._h, B, _ptr(state), _ptr(k_coeffs), _ptr(v_des), _ptr(u_prev), _ptr(warm),
                                                         _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj), HOST))
        else:
            w = _weight_rows(weights, B, 7, "solve_batch")
            self._check(lib().mpcb200_solve_batch_frenet_w(self._h, B, _ptr(state), _ptr(k_coeffs), _ptr(v_des), _ptr(u_prev), _ptr(warm),
                                                           _ptr(w), _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj), HOST))
        return {"u0": u0, "cost": cost, "status": status, "iters": iters, "traj": traj}

    def rollout(self, pose0, path_of, T, window=40.0, target_vel=8.0, ey_from_path=True, want_log=True, metrics=False, weights=None):
        """Closed loop on the Frenet-frame module on the device (mpcb200_rollout_frenet; what closed_loop.run_frenet does on the
        host).  pose0 (B,3); path_of (B,) ids given to set_path.  Returns log (T,B,8) and final (B,8) like Solver.rollout;
        metrics: also out["metrics"] (B,12) as Solver.rollout (mpcb200_rollout_frenet_metrics).
        weights (B,7) in set_cost's order (cey, cep, cev, cda, cdd, ca, cd): each vehicle's cost weights for all its control
        periods (mpcb200_rollout_frenet_w, with or without metrics), or None: the handle's."""
        pose0 = np.ascontiguousarray(np.atleast_2d(pose0), dtype=np.float64)
        B = pose0.shape[0]
        path_of = np.ascontiguousarray(path_of, dtype=np.int32)
        if pose0.shape != (B, 3) or path_of.shape != (B,):
            raise ValueError("rollout: pose0 must be (B,3) and path_of (B,)")
        log = np.empty((T, B, 8)) if want_log else None
        final = np.empty((B, 8))
        dp = C.POINTER(C.c_double)
        args = [pose0.ctypes.data_as(dp), path_of.ctypes.data_as(C.POINTER(C.c_int32)), float(window), float(target_vel),
                int(bool(ey_from_path)), None if log is None else log.ctypes.data_as(dp), final.ctypes.data_as(dp)]
        if weights is not None:
            w = _weight_rows(weights, B, 7, "rollout")
            met = np.empty((B, len(ROLLOUT_METRICS))) if metrics else None
            self._check(lib().mpcb200_rollout_frenet_w(self._h, B, int(T), *args[:5], w.ctypes.data_as(dp), *args[5:],
                                                       None if met is None else met.ctypes.data_as(dp)))
            out = {"log": log, "final_state": final}
            if metrics:
                out["metrics"] = met
            return out
        if metrics:
            met = np.empty((B, len(ROLLOUT_METRICS)))
            self._check(lib().mpcb200_rollout_frenet_metrics(self._h, B, int(T), *args, met.ctypes.data_as(dp)))
            return {"log": log, "final_state": final, "metrics": met}
        self._check(lib().mpcb200_rollout_frenet(self._h, B, int(T), *args))
        return {"log": log, "final_state": final}

    def solve_batch_on_path(self, pose, path_of, u_prev, window=40.0, target_vel=8.0, ey_from_path=True, v_des=None, warm=None,
                            want_traj=False, want_ref=False, weights=None):
        """mpcb200_solve_batch_frenet_on_path: the node's reference step (nearest sample, the next `window` metres of the path set
        with set_path, the curvature fit, psi_start, e_y) on the device from each pose, then the solve.  pose (B,4) = X, Y, psi, v;
        path_of (B,) ids given to set_path; v_des (B,) or None = target_vel; warm, weights as in solve_batch.  Returns the
        solve_batch dict; with want_ref also "k_coeffs" (B,4) and "state" (B,4) = (0, e_y, -psi_start, v), the solver's inputs."""
        N = self.N
        pose = np.ascontiguousarray(pose, dtype=np.float64)
        B = pose.shape[0]
        path_of = np.ascontiguousarray(path_of, dtype=np.int32)
        u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
        if pose.shape != (B, 4) or path_of.shape != (B,) or u_prev.shape != (B, 2):
            raise ValueError("solve_batch_on_path: expected pose (B,4), path_of (B,), u_prev (B,2)")
        if v_des is not None:
            v_des = np.ascontiguousarray(v_des, dtype=np.float64)
            if v_des.shape != (B,):
                raise ValueError("solve_batch_on_path: v_des must be (B,)")
        if warm is not None:
            if not (isinstance(warm, np.ndarray) and warm.dtype == np.float64 and warm.flags.c_contiguous
                    and warm.shape == (B, 6 * N + 4)):
                raise ValueError("solve_batch_on_path: warm must be a C-contiguous float64 (B,6N+4) array (updated in place)")
        w = None if weights is None else _weight_rows(weights, B, 7, "solve_batch_on_path")
        u0 = np.empty((B, 2)); cost = np.empty(B)
        status = np.empty(B, dtype=np.int32); iters = np.empty(B, dtype=np.int32)
        traj = np.empty((B, 6 * N + 4)) if want_traj else None
        k_coeffs = np.empty((B, 4)) if want_ref else None
        state = np.empty((B, 4)) if want_ref else None
        self._check(lib().mpcb200_solve_batch_frenet_on_path(self._h, B, _ptr(pose), _ptr(path_of), float(window), float(target_vel),
                                                             int(bool(ey_from_path)), _ptr(v_des), _ptr(u_prev), _ptr(warm), _ptr(w),
                                                             _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj),
                                                             _ptr(k_coeffs), _ptr(state), HOST))
        out = {"u0": u0, "cost": cost, "status": status, "iters": iters, "traj": traj}
        if want_ref:
            out["k_coeffs"] = k_coeffs
            out["state"] = state
        return out

    def solve_batch_on_path_device(self, B, pose, path_of, u_prev, u0, window=40.0, target_vel=8.0, ey_from_path=True, v_des=None,
                                   warm=None, cost=None, status=None, iters=None, traj=None, k_coeffs_out=None, state_out=None,
                                   weights=None):
        """solve_batch_on_path with device pointers (torch CUDA tensors, float64 / int32, contiguous); only enqueues on the
        handle's stream.  An unset path id or a bad weight row gives that problem status ERROR (and, for the path id, NaN rows in
        k_coeffs_out / state_out)."""
        w = None if weights is None else _weight_rows_device(weights, B, 7, "solve_batch_on_path_device")
        self._check(lib().mpcb200_solve_batch_frenet_on_path(self._h, B, _ptr(pose), _ptr(path_of), float(window), float(target_vel),
                                                             int(bool(ey_from_path)), _ptr(v_des), _ptr(u_prev), _ptr(warm), _ptr(w),
                                                             _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj),
                                                             _ptr(k_coeffs_out), _ptr(state_out), DEVICE))

    def solve_batch_device(self, B, state, k_coeffs, u_prev, u0, v_des=None, warm=None, cost=None, status=None, iters=None, traj=None,
                           weights=None):
        """Device pointers (torch CUDA tensors or ints); asynchronous on the handle's stream.  weights: (B,7) float64 tensor, one row
        per problem (a bad row gives that problem status ERROR), or None: the handle's weights."""
        if weights is None:
            self._check(lib().mpcb200_solve_batch_frenet(self._h, B, _ptr(state), _ptr(k_coeffs), _ptr(v_des), _ptr(u_prev), _ptr(warm),
                                                         _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj), DEVICE))
        else:
            w = _weight_rows_device(weights, B, 7, "solve_batch_device")
            self._check(lib().mpcb200_solve_batch_frenet_w(self._h, B, _ptr(state), _ptr(k_coeffs), _ptr(v_des), _ptr(u_prev), _ptr(warm),
                                                           _ptr(w), _ptr(u0), _ptr(cost), _ptr(status), _ptr(iters), _ptr(traj), DEVICE))
