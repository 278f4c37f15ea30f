/*
 * mpc_b200.h -- C ABI of libmpc_b200.so, the B200-native batched solver for the
 * kinematic-bicycle path-following NLP.
 *
 * Drop-in boundary.  The reference has no FFI layer; its boundary is the Julia module
 * API of scripts/mpc_utils/MKZMPCPathFollower.jl as called from scripts/mpc_cmd_pub.jl.
 * Each entry point below names the reference interface it replaces.  A Julia shim
 * (julia/MKZMPCPathFollower.jl, ccall) and a Python ctypes binding
 * (mkz_mpc_path_follower_b200/capi.py) sit on top; see INTEGRATION.md.
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative
 * MPCB200_E* code (message via mpcb200_last_error); the caller owns every buffer, the
 * library owns the opaque handle, its device scratch and its CUDA stream(s).  Calls on one
 * handle must be serialised by the caller; distinct handles are independent.  There is
 * no CPU fallback: without a CUDA device mpcb200_create fails with MPCB200_ENODEVICE.
 *
 * Multi-GPU (SURVEY.md 8b/8e): a handle created with n_devices > 1 owns one stream and one set of
 * device buffers per GPU.  Calls with HOST pointers (mpcb200_solve_batch*, mpcb200_rollout) cut the
 * batch into contiguous slices, one per device, run them concurrently and write every slice's
 * results straight into the caller's one set of buffers -- problems are independent, nothing
 * crosses GPUs, and the results do not depend on the device count.  Calls with DEVICE pointers and
 * batches of at most 64 problems run on devices[0].  (Multi-process use, one rank per GPU under
 * torchrun, gathers mpcb200_solve_batch_records' 32-byte records with one NCCL all-gather instead.)
 */
#ifndef MPC_B200_H
#define MPC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPCB200_VERSION 6

/* error codes */
#define MPCB200_OK          0
#define MPCB200_EINVAL     -1  /* bad argument (NULL pointer, N out of range, B < 0, ...) */
#define MPCB200_ENODEVICE  -2  /* no usable CUDA device: the library has no CPU path */
#define MPCB200_ECUDA      -3  /* CUDA runtime error, text in mpcb200_last_error */
#define MPCB200_ENOMEM     -4

/* solve status, one per problem: the JuMP status symbols solve_model() returns
 * (MKZMPCPathFollower.jl:176-182) through Ipopt.jl's mapping */
#define MPCB200_OPTIMAL     0  /* :Optimal    Solve_Succeeded / Solved_To_Acceptable_Level */
#define MPCB200_INFEASIBLE  1  /* :Infeasible */
#define MPCB200_UNBOUNDED   2  /* :Unbounded  diverging iterates */
#define MPCB200_USERLIMIT   3  /* :UserLimit  iteration cap (stands in for max_cpu_time, :29) */
#define MPCB200_ERROR       4  /* :Error      everything else */

/* mem_space */
#define MPCB200_HOST   0  /* pointers are host memory; the call copies H2D/D2H and synchronises */
#define MPCB200_DEVICE 1  /* pointers are device memory on the handle's device; the call only
                             enqueues work on the handle's stream (no synchronisation) */

/* start_mode when warm == NULL */
#define MPCB200_START_ZERO    0  /* every variable 0.0, as `start=0.0` in MKZMPCPathFollower.jl:65-72 */
#define MPCB200_START_ROLLOUT 1  /* states = bicycle-model rollout of the previous command from the
                                    measured state (not a reference behaviour; opt-in) */

/* Replaces the module-level constants of MKZMPCPathFollower.jl:28-48.  mpcb200_create refuses (MPCB200_EINVAL, the message
 * names the field) a constant that is not finite, dt, dt_control, L_b, a_max, a_dmax, steer_dmax or tol <= 0, L_a < 0,
 * v_max <= v_min, steer_max outside (0, 1.5) and max_iter < 0.
 * tol: supported up to 1e-5.  Above that, Ipopt's barrier floor min(tol, 1e-4) / 11 (in the scaled problem) can lie above the
 * unscaled complementarity tolerance 1e-4, and a solve that has reached the optimum of that barrier problem ends with
 * MPCB200_ERROR (Ipopt: Search_Direction_Becomes_Too_Small), or UserLimit, instead of Optimal (DESIGN.md section 5). */
typedef struct {
    int32_t N;            /* horizon (:34), 3 <= N <= 95: one warp per problem up to 31, one block of 2-3 warps beyond */
    int32_t max_iter;     /* iteration cap -> MPCB200_USERLIMIT */
    int32_t start_mode;   /* MPCB200_START_* */
    int32_t device;       /* CUDA device ordinal */
    double  dt;           /* :33 */
    double  dt_control;   /* :28 */
    double  L_a, L_b;     /* :31-32 */
    double  v_min, v_max; /* :47-48 */
    double  a_max;        /* :44 */
    double  steer_max;    /* :41 */
    double  a_dmax;       /* :45 */
    double  steer_dmax;   /* :42 */
    double  tol;          /* Ipopt tol, default 1e-8 */
    int32_t n_devices;    /* 0 or 1: one GPU, `device`.  2..8: the GPUs devices[0..n_devices-1] (`device` is ignored) */
    int32_t devices[8];   /* CUDA device ordinals, distinct */
} mpcb200_config;

typedef struct mpcb200_handle mpcb200_handle;

/* Fill *cfg with the reference's constants (MKZMPCPathFollower.jl:28-48) for horizon N. */
int mpcb200_default_config(mpcb200_config* cfg, int32_t N);

/* Replaces module load (`import MKZMPCPathFollower`, mpc_cmd_pub.jl:45-47): builds the solver
 * for one horizon on one GPU.  Weights start at the module defaults (:51-59). */
int mpcb200_create(mpcb200_handle** out, const mpcb200_config* cfg);
int mpcb200_destroy(mpcb200_handle* h);

/* Replaces update_cost(cx, cy, cp, cv, cda, cdd, ca, cd) (MKZMPCPathFollower.jl:158-169);
 * same argument order. */
int mpcb200_set_cost(mpcb200_handle* h, const double w[8]);

/* Use an existing CUDA stream (cudaStream_t passed as void*) for all work of this handle;
 * NULL restores the handle's own stream. */
int mpcb200_set_stream(mpcb200_handle* h, void* cuda_stream);

/* Which kernel solves mpcb200_solve_batch / _records / _on_path batches of the XY model (no reference counterpart: the reference
 * solves one problem at a time, MKZMPCPathFollower.jl:176).  Two device layouts of the same solver exist: one warp per
 * problem with the iterate on chip (every batch size, lowest latency) and one THREAD per problem with the iterate
 * streamed from HBM (csrc/tpp_solver.cuh: faster for large batches at short horizons, e.g. 1.5x at 65,536 problems and
 * 2.1x at 262,144 problems for N = 8; slower for N >= 12 below ~131,072 problems).  Both follow the same iteration and
 * agree to rounding, not bit for bit.
 *   min_batch  > 0: batches (per device) of at least min_batch problems use one thread per problem
 *   min_batch == 0: always one warp per problem
 *   min_batch  < 0: the default rule, what a new handle starts with.  XY model: N <= 10: 32,768, and 16,384 for warm-started or
 *                   rollout-started batches, whose solves all take about the same handful of iterations; N > 10: never.
 *                   Frenet-frame handles (every solve takes 14-17 iterations): 16,384 at N <= 10, 32,768 at longer horizons
 *                   (N = 20, 65,536 problems: 4.8 M instead of 3.2 M solves/s)
 * mpcb200_solve_batch_on_path follows the switch for N <= 31: the waypoints of the batch are generated by a kernel of their own
 * (same generator, same bits), then the thread-per-problem solve, then the answers of problems with an unknown path id: three
 * launches (N = 8, host buffers, whole call: 3.3 M instead of 1.9 M solves/s at 65,536 problems, 4.1 M at 262,144).
 * mpcb200_rollout and mpcb200_rollout_frenet follow the same switch: fleets of at least min_batch vehicles per device (default rule:
 * a quarter of the batch rule, i.e. 8,192 vehicles at N <= 10 for the XY model, 4,096 for the Frenet node) run
 * each control period as three launches over the whole fleet -- plant, waypoints, thread-per-problem solve warm-started in place
 * -- instead of one persistent kernel (16,384 vehicles x 500 periods: 0.64 s instead of 1.38 s; 65,536 x 100: 0.38 s instead of
 * 1.39 s). */
int mpcb200_set_large_batch_path(mpcb200_handle* h, int64_t min_batch);

/*
 * Replaces, for B independent problems at once, the per-step sequence of mpc_cmd_pub.jl:115-141:
 *   update_init_cond(x, y, psi, v)                 -> state  [B][4]
 *   update_reference(x_ref, y_ref, psi_ref, v_des) -> ref    [B][3][N+1]  and v_des [B] (NULL = 0)
 *   update_current_input(c_swa, c_acc)             -> u_prev [B][2]   (steering first, :151)
 *   solve_model() -> (acc, d_f, status)            -> u0     [B][2]   (acceleration first, :182),
 *                                                     status [B], plus cost [B] and iters [B]
 *   get_solver_results()                           -> traj   [B][6N+4] in the order
 *        x[N+1], y[N+1], v[N+1], psi[N+1], d_f[N], acc[N]   (:188-206); may be NULL
 * warm [B][6N+4] (same layout as traj): in = start point (the reference re-solves from the
 * previous solution), out = this solution.  NULL = start_mode of the config.
 * cost, status, iters, traj, warm may each be NULL.  All problem-major, contiguous.
 */
int mpcb200_solve_batch(mpcb200_handle* h, int64_t B,
                        const double* state, const double* ref, const double* v_des,
                        const double* u_prev, double* warm,
                        double* u0, double* cost, int32_t* status, int32_t* iters,
                        double* traj, int32_t mem_space);

/*
 * mpcb200_solve_batch with one cost-weight row per problem: w [B][8] in update_cost order (cx, cy, cp, cv, cda, cdd, ca, cd),
 * so one batch can hold controllers with different tunings (a weight sweep is one call).  The handle's own weights
 * (mpcb200_set_cost) are neither used nor changed by this call.  A weight is valid by mpcb200_set_cost's rule (not negative, not
 * NaN): with MPCB200_HOST pointers a bad row is refused (MPCB200_EINVAL, the message names the problem and the weight index); with
 * MPCB200_DEVICE pointers that problem alone comes back with MPCB200_ERROR, zero commands, cost 0, 0 iterations and 0 restorations.
 * Everything else -- both device layouts (mpcb200_set_large_batch_path), multi-GPU slicing, the small-batch path,
 * mpcb200_get_stats and mpcb200_get_restorations -- as in mpcb200_solve_batch.  w is required.
 */
int mpcb200_solve_batch_w(mpcb200_handle* h, int64_t B, const double* state, const double* ref, const double* v_des,
                          const double* u_prev, double* warm, const double* w,
                          double* u0, double* cost, int32_t* status, int32_t* iters, double* traj, int32_t mem_space);

/*
 * mpcb200_solve_batch whose per-problem results come back as ONE packed 32-byte record
 *   rec [B][4] doubles = { accel_cmd, steer_angle_cmd, cost, (int32 status | restorations << 8, int32 iters) }
 * written by the solve kernel itself: the unit of the multi-GPU exchange (one all-gather of these records is the only
 * inter-GPU traffic, SURVEY.md 8e).  `restorations` = how many times the solve went through the restoration by rollout
 * that stands in for Ipopt's restoration phase (0 for almost every problem).  traj and warm as in mpcb200_solve_batch.
 */
int mpcb200_solve_batch_records(mpcb200_handle* h, int64_t B,
                                const double* state, const double* ref, const double* v_des,
                                const double* u_prev, double* warm, double* rec, double* traj, int32_t mem_space);

/* Per-problem restoration counts of the LAST solve_batch* call on this handle (host pointer, B = that call's batch):
 * the problems whose line search failed where Ipopt would enter its restoration phase (MKZMPCPathFollower.jl:176). */
int mpcb200_get_restorations(mpcb200_handle* h, int64_t B, int32_t* out);

/* Path table for on-device reference generation (ref_gps_traj.py:106): columns t, X, Y, psi, s
 * of the trajectory matrix, n samples each, host pointers; copied to the device. */
int mpcb200_set_path(mpcb200_handle* h, int32_t path_id, int32_t n,
                     const double* t, const double* X, const double* Y,
                     const double* psi, const double* s);

/*
 * mpcb200_solve_batch with the waypoints generated ON THE DEVICE from the path tables: replaces, per
 * problem, grt.get_waypoints(x, y, psi[, des_speed]) of mpc_cmd_pub.jl:99-112 (ref_gps_traj.py:131-218:
 * nearest sample over the whole path, np.interp of X, Y, psi at t_closest + h*dt -- or at
 * s_closest + (h+1)*dt*target_vel when !track_using_time --, heading unwrap, stop_cmd) followed by the
 * update_* / solve_model sequence above.  Input shrinks from 3(N+1)+7 to 7 doubles + one int per problem.
 *   path_of [B]  path_id (0..2) given to mpcb200_set_path
 *   v_des   [B] or NULL = target_vel for every problem (mpc_cmd_pub.jl:116 passes des_speed)
 *   ref_out [B][3][N+1] or NULL: the generated waypoints (what the node publishes as target_path)
 *   stop    [B] or NULL: get_waypoints' stop_cmd (1 when the last waypoint is the end of the path)
 * With MPCB200_HOST pointers a path_of entry that was not set is refused (MPCB200_EINVAL); with MPCB200_DEVICE pointers
 * the ids cannot be inspected on the host: such a problem comes back with status MPCB200_ERROR and zero commands.
 */
int mpcb200_solve_batch_on_path(mpcb200_handle* h, int64_t B,
                                const double* state, const int32_t* path_of,
                                int32_t track_using_time, double target_vel,
                                const double* v_des, const double* u_prev, double* warm,
                                double* u0, double* cost, int32_t* status, int32_t* iters,
                                double* traj, double* ref_out, int32_t* stop, int32_t mem_space);

/*
 * Closed-loop Monte-Carlo rollout (mpc_cmd_pub.jl:86-157 driving vehicle_simulator.py:58-112):
 * B vehicles x T control steps, each step = 10 plant publishes (100 Euler sub-steps), on-device
 * reference generation (time mode if target_vel <= 0 ... see track_using_time), warm-started solve,
 * command feedback, stop latch.
 *   pose0    [B][3]  X0, Y0, Psi0 ;  path_of [B] path_id per vehicle
 *   log      [T][B][8]  x, y, psi, v, acc_cmd, df_cmd, status, iters  (may be NULL)
 *   final    [B][8]  plant state X,Y,psi,vx,vy,wz,acc,df after T steps (may be NULL)
 * Every vehicle's first solve starts from the solution of the module-load solve of the default problem
 * (MKZMPCPathFollower.jl:36-39,126-128), as the node's does.  Host pointers only; any horizon the handle supports;
 * vehicles are sharded over the handle's devices.
 */
int mpcb200_rollout(mpcb200_handle* h, int64_t B, int32_t T,
                    const double* pose0, const int32_t* path_of,
                    int32_t track_using_time, double target_vel,
                    double* log, double* final_state);

/* mpcb200_rollout with one cost-weight row per vehicle, w [B][8] in update_cost order, used in every control period of that
 * vehicle (a closed-loop tuning sweep in one call).  Rows are checked as by mpcb200_solve_batch_w with host pointers.  The first
 * solve of every vehicle still starts from the module-load solution of the default problem (the node loads the module before any
 * update_cost).  Host pointers only; same kernels, same fused / per-period switch and same sharding as mpcb200_rollout. */
int mpcb200_rollout_w(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of,
                      int32_t track_using_time, double target_vel, const double* w, double* log, double* final_state);

/*
 * Tracking metrics of a closed-loop rollout, accumulated on the device while it runs (the offline score of
 * scripts/analysis/plot_path_tracking_error.py -- nearest-sample path error and heading error -- plus command smoothness, solver
 * health and progress), so that scoring a large sweep needs neither the [T][B][8] log nor a host-side nearest-sample search.
 * metrics [B][MPCB200_METRICS] is required; everything else -- validation, w ([B][8] rows as mpcb200_rollout_w, or NULL = the
 * handle's weights), host pointers, the fused / per-period switch, multi-GPU slicing, log and final_state (either may be NULL) --
 * is that of mpcb200_rollout / mpcb200_rollout_w, and log and final_state come out bit-identical to theirs.
 *
 * A period COUNTS when a solve ran in it (log status >= 0): every period before the stop latch (the period in which stop_cmd
 * latches does not count).  For the pose (x, y, psi) logged for that period and its nearest path sample i (the one get_waypoints
 * uses): e = sqrt((X_i - x)^2 + (Y_i - y)^2), h = mod(psi - psi_i + pi, 2 pi) - pi, and the command rates
 * da = acc_cmd - acc_cmd_prev, dd = df_cmd - df_cmd_prev, "prev" being the previous counting period's command (0 for the first).
 * Per vehicle, in this order (n = field 0; with n = 0 fields 1..9 are 0):
 *    0 n_solved         counting periods             6 acc_rate_rms    sqrt(sum da^2 / n)
 *    1 path_err_mean    sum e / n                    7 steer_rate_rms  sqrt(sum dd^2 / n)
 *    2 path_err_rms     sqrt(sum e^2 / n)            8 n_not_optimal   counting periods with status != MPCB200_OPTIMAL
 *    3 path_err_max     max e                        9 iters_total     sum of iterations
 *    4 heading_err_rms  sqrt(sum h^2 / n)           10 s_last          arc length s_i of the last counting period (NaN if n = 0)
 *    5 heading_err_max  max |h|                     11 stop_period     first period with status -1 (stop latch), -1 if none
 * Every operation is rounded as numpy rounds it and the sums run in period order: closed_loop.tracking_metrics restates this on
 * the host from a log.  metrics == NULL is MPCB200_EINVAL; with B == 0 or T == 0 nothing is written.
 */
#define MPCB200_METRICS 12   /* doubles per vehicle */
int mpcb200_rollout_metrics(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of,
                            int32_t track_using_time, double target_vel, const double* w,
                            double* log, double* final_state, double* metrics);

/*
 * Frenet-frame variant of the same solver: scripts/mpc_utils/MKZMPCPathFollowerFrenet.jl (the model the Gazebo
 * lane-keep node gazebo_sim_mpc_cmd_pub_frenet.jl:112-153 drives).  Same vehicle constants, horizon, bounds, rate
 * rows and interior-point iteration; states (s, e_y, e_psi, v) with ds/dt = v cos(e_psi + beta) / (1 - e_y K(s)),
 * K(s) a cubic (:111-120); cost on e_y, e_psi, v - v_target and the input terms (:95-101).
 *   mpcb200_create_frenet            replaces module load (:28-129); 3 <= N <= 95; weights start at (:51-58)
 *   mpcb200_set_cost_frenet          replaces update_cost(cey, cep, cev, cda, cdd, ca, cd) (:158-169), same order
 *   mpcb200_solve_batch_frenet       replaces, for B problems at once,
 *       update_init_cond(s, ey, epsi, vel) (:132-138)        -> state    [B][4]
 *       update_reference(path, k_coeffs, v_des) (:142-147)   -> k_coeffs [B][4] (highest degree first, :40-41), v_des [B]
 *       update_current_input(c_swa, c_acc) (:151-154)        -> u_prev   [B][2]
 *       solve_model() (:173-183)                             -> u0 [B][2] (acc, d_f), status, cost, iters
 *       get_solver_results() (:188-207)                      -> traj [B][6N+4] = s[N+1], ey[N+1], v[N+1], epsi[N+1], d_f[N], acc[N]
 *   warm as in mpcb200_solve_batch.  mpcb200_solve_batch / _on_path / _rollout refuse a Frenet handle; the Frenet form of
 *   _on_path is mpcb200_solve_batch_frenet_on_path below.
 */
int mpcb200_create_frenet(mpcb200_handle** out, const mpcb200_config* cfg);
int mpcb200_set_cost_frenet(mpcb200_handle* h, const double w[7]);
int mpcb200_solve_batch_frenet(mpcb200_handle* h, int64_t B, const double* state, const double* k_coeffs,
                               const double* v_des, const double* u_prev, double* warm, double* u0,
                               double* cost, int32_t* status, int32_t* iters, double* traj, int32_t mem_space);
/* mpcb200_solve_batch_frenet with one cost-weight row per problem: w [B][7] in the update_cost order of
 * MKZMPCPathFollowerFrenet.jl (cey, cep, cev, cda, cdd, ca, cd); validation and everything else as mpcb200_solve_batch_w. */
int mpcb200_solve_batch_frenet_w(mpcb200_handle* h, int64_t B, const double* state, const double* k_coeffs,
                                 const double* v_des, const double* u_prev, double* warm, const double* w,
                                 double* u0, double* cost, int32_t* status, int32_t* iters, double* traj, int32_t mem_space);

/*
 * Closed loop on the Frenet-frame module, on the device (scripts/nodes_gazebo_sim/gazebo_sim_mpc_cmd_pub_frenet.jl:112-153
 * around the plant of scripts/vehicle_simulator.py:58-112; Gazebo itself is out of scope): B vehicles x T control steps.
 * Per step and vehicle: the next `window` metres of its path (mpcb200_set_path) from the sample nearest to the vehicle,
 * seen from the vehicle -> K_coeffs, psi_start = get_reference_frenet (scripts/sim_path_utils/nav_msgs_path_frenet.py:44-86:
 * two cubic least-squares fits on fixed grids) -> update_init_cond(0, e_y, -psi_start, v) (:125; e_y = 0 like the node, or
 * the vehicle's lateral offset from the fitted path start when ey_from_path != 0), update_reference(path, K_coeffs,
 * target_vel) (:126), solve_model from the previous solution (:130), command published whatever the status (:139-143),
 * update_current_input(df_opt, a_opt) (:145).  log / final as in mpcb200_rollout.  Frenet handles, N <= 31, host pointers.
 */
int mpcb200_rollout_frenet(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of,
                           double window, double target_vel, int32_t ey_from_path, double* log, double* final_state);
/* mpcb200_rollout_frenet with the tracking metrics of mpcb200_rollout_metrics (every period counts; stop_period is always -1).
 * mpcb200_rollout_metrics refuses a Frenet handle (MPCB200_EINVAL); per-vehicle weights are mpcb200_rollout_frenet_w's. */
int mpcb200_rollout_frenet_metrics(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of,
                                   double window, double target_vel, int32_t ey_from_path,
                                   double* log, double* final_state, double* metrics);
/* mpcb200_rollout_frenet with one cost-weight row per vehicle, w [B][7] in the update_cost order of MKZMPCPathFollowerFrenet.jl
 * (cey, cep, cev, cda, cdd, ca, cd), used in every control period of that vehicle (a Frenet closed-loop tuning sweep in one call).
 * w is required (NULL with B > 0 and T > 0 is MPCB200_EINVAL); rows are checked as by mpcb200_solve_batch_frenet_w with host
 * pointers.  metrics [B][MPCB200_METRICS] or NULL: when given, filled as mpcb200_rollout_frenet_metrics fills it.  Everything else
 * -- host pointers, N <= 31, window, the fused / per-period switch, the first solve from all zeros, devices[0] of a multi-GPU
 * handle -- is that of mpcb200_rollout_frenet. */
int mpcb200_rollout_frenet_w(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of,
                             double window, double target_vel, int32_t ey_from_path, const double* w,
                             double* log, double* final_state, double* metrics);

/*
 * Frenet-frame batch from vehicle poses, the open-loop form of one period of mpcb200_rollout_frenet: for each problem the node's
 * reference step (gazebo_sim_mpc_cmd_pub_frenet.jl:112-130 with nav_msgs_path_frenet.py:44-86: nearest path sample, the next
 * `window` metres resampled every 0.5 m in the vehicle frame, cubic fits of X(s) and Y(s), their curvature every 0.25 m fitted
 * by a cubic, psi_start and e_y) computed on the device exactly as mpcb200_rollout_frenet computes it, then the solve.  Replaces
 * the node's get_reference_frenet + update_init_cond / update_reference / update_current_input + solve_model sequence.
 *   pose          [B][4]  X, Y, psi, v (the node's state_est)
 *   path_of       [B]     path ids given to mpcb200_set_path
 *   window        length of the path ahead in metres, in [4, 500]; target_vel, ey_from_path as in mpcb200_rollout_frenet
 *   v_des         [B] or NULL = target_vel for every problem
 *   u_prev, warm, u0, cost, status, iters, traj as in mpcb200_solve_batch_frenet
 *   w             [B][7] Frenet weight rows as in mpcb200_solve_batch_frenet_w, or NULL = the handle's weights
 *   k_coeffs_out  [B][4] or NULL: K(s), highest degree first
 *   state_out     [B][4] or NULL: (0, e_y, -psi_start, v) as given to the solver
 * u0, cost, status, iters, traj and warm are bit-identical to those of mpcb200_solve_batch_frenet (or _w with w) called with the
 * returned state_out and k_coeffs_out: the solve is the same kernel in the same layout on those rows.  pose, path_of, u_prev and
 * u0 are required; any horizon of a Frenet handle; host pointers are sliced over a multi-GPU handle like every host solve call,
 * device pointers run on devices[0].  A handle from mpcb200_create and a window outside [4, 500] (or NaN) are MPCB200_EINVAL.
 * With MPCB200_HOST pointers an unset path id or a negative or NaN weight is refused (MPCB200_EINVAL, naming the problem); with
 * MPCB200_DEVICE pointers that problem alone comes back with status MPCB200_ERROR, zero commands, cost 0 and 0 iterations, and
 * for an unset path id NaN in its k_coeffs_out and state_out rows.  Three kernel launches (reference, solve, answers for unset ids).
 */
int mpcb200_solve_batch_frenet_on_path(mpcb200_handle* h, int64_t B, const double* pose, const int32_t* path_of,
                                       double window, double target_vel, int32_t ey_from_path,
                                       const double* v_des, const double* u_prev, double* warm, const double* w,
                                       double* u0, double* cost, int32_t* status, int32_t* iters, double* traj,
                                       double* k_coeffs_out, double* state_out, int32_t mem_space);

/* Counters of the last solve_batch/rollout call on this handle. */
typedef struct {
    int64_t kernel_launches;   /* kernels of this library launched by the call (a radix sort counts as one) */
    int64_t h2d_bytes, d2h_bytes;
    float   kernel_ms;         /* device time of the solver kernel(s) (CUDA events), HOST mode only */
} mpcb200_stats;
int mpcb200_get_stats(mpcb200_handle* h, mpcb200_stats* out);

/* FP64 FMA micro-benchmark on the handle's device: returns achieved TFLOP/s (2 flop per FMA).
 * Used for the roofline denominator (MEASURED_PEAKS.json has no FP64 entry). */
int mpcb200_fp64_peak(mpcb200_handle* h, double* tflops);

const char* mpcb200_last_error(mpcb200_handle* h);
int mpcb200_version(void);

#ifdef __cplusplus
}
#endif
#endif
