// mpc_b200.cu -- C ABI (include/mpc_b200.h) and kernel launches for sm_100a.
//
// One handle = one GPU + one stream.  Problems are independent: a persistent grid of warps
// pulls problem indices from a device counter (iteration counts differ per problem, so a
// dynamic queue keeps the SMs level), solves each with mpc_kernel.cuh::solve_problem and
// writes the per-problem record.  No CPU path exists in this library.
#include "../../include/mpc_b200.h"
#include "mpc_kernel.cuh"
#include "tpp_solver.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <utility>

using namespace mpcb200;
static_assert(MET_FIELDS == MPCB200_METRICS, "rollout metrics: kernel and C ABI row sizes differ");

namespace {

constexpr int WARPS_PER_BLOCK = 4;

// 168 registers per thread: three blocks (12 warps) per SM at the N = 20 shared-memory footprint.
// The iterate's bound multipliers, the step and the model evaluation live in per-thread shared-memory
// fields (mpc_kernel.cuh, LF_*), which is what lets the solver fit.
//
// PW (every solve kernel below): 1 = each problem's cost weights from io.w (mpcb200_solve_batch_w / _frenet_w), 0 = KCfg::w.
// A compile-time switch, so that the PW = 0 instantiations the unweighted entry points launch are the code they always were.
#ifndef MPC_MIN_BLOCKS
#define MPC_MIN_BLOCKS 3
#endif
#ifndef MPC_ORDER_MIN_QUARTER_WAVES
#define MPC_ORDER_MIN_QUARTER_WAVES 5   /* mpcb200_create: from how many quarter waves of resident teams a batch is ordered (0: all) */
#endif
//
// ORD = 1: the queue is `order` (a permutation of 0 .. B-1, longest predicted solve first: queue_key_kernel and a radix sort),
// and a warp solves problem order[counter] instead of problem counter.  Every problem still reads and writes its own index, so
// the results are those of ORD = 0 bit for bit; only which warp solves a problem, and when, changes.  The team kernels take
// `order` as their last parameter so that they share one launch signature; the ORD = 0 builds never read it.
template <int PW, int ORD = 0>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, MPC_MIN_BLOCKS)
mpc_solve_kernel(const KCfg cfg, const BatchPtrs io, const RefGen rg, const long long B, unsigned long long* counter, const int* order) {
    extern __shared__ double smem_all[];
    const int warp = threadIdx.x >> 5;
    const smem_t smem = smem_base(smem_all + (size_t)warp * smem_doubles_per_team(cfg.N, 0, PW));
    TeamSolver<1>::init_work(smem, cfg.N);
    for (;;) {
        unsigned long long b = 0;
        if ((threadIdx.x & 31) == 0) {
            b = atomicAdd(counter, 1ULL);
            if (ORD && b < (unsigned long long)B) b = (unsigned long long)order[b];
        }
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= (unsigned long long)B) break;
        solve_problem<1, 0, PW>(cfg, io, rg, (long)b, smem);
        __syncwarp();
    }
}

// Frenet-frame variant (MKZMPCPathFollowerFrenet.jl): same driver, dense s / e_y columns (mpc_kernel.cuh, MODEL 1);
// 62-double records, 21.3 KB of shared memory per problem at N = 20.  Two builds: blocks of four warps at 255 registers
// (two per SM) and blocks of three at 168 registers with spill code (up to four per SM: 12 warps at the N = 8 footprint);
// mpcb200_create_frenet picks per horizon (see there)
template <int WPB, int PW = 0>
__global__ void __launch_bounds__(WPB * 32, WPB == 3 ? 3 : 2)
mpc_solve_frenet_kernel(const KCfg cfg, const BatchPtrs io, const RefGen rg, const long long B, unsigned long long* counter, const int*) {
    extern __shared__ double smem_all[];
    const int warp = threadIdx.x >> 5;
    const smem_t smem = smem_base(smem_all + (size_t)warp * smem_doubles_per_team(cfg.N, 1, PW));
    TeamSolver<1, 1>::init_work(smem, cfg.N);
    for (;;) {
        unsigned long long b = 0;
        if ((threadIdx.x & 31) == 0) b = atomicAdd(counter, 1ULL);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= (unsigned long long)B) break;
        solve_problem<1, 1, PW>(cfg, io, rg, (long)b, smem);
        __syncwarp();
    }
}

// Long horizons (32 <= N <= 95): one problem per block of W = 2 or 3 warps, thread k = stage k.
// register budget (measured at N = 40 / 80): W = 2 -> 6 blocks (12 warps) per SM at 168 registers; W = 3 -> 2 blocks at 255
#ifndef MPC_LONG_MIN_BLOCKS2
#define MPC_LONG_MIN_BLOCKS2 6
#define MPC_LONG_MIN_BLOCKS3 2
#endif
template <int W, int MODEL = 0, int PW = 0>
__global__ void __launch_bounds__(W * 32, MODEL ? 2 : (W == 2 ? MPC_LONG_MIN_BLOCKS2 : MPC_LONG_MIN_BLOCKS3))
mpc_solve_long_kernel(const KCfg cfg, const BatchPtrs io, const RefGen rg, const long long B, unsigned long long* counter, const int*) {
    extern __shared__ double smem_all[];
    __shared__ unsigned long long next_problem;
    const smem_t smem = smem_base(smem_all);
    TeamSolver<W, MODEL>::init_work(smem, cfg.N);
    for (;;) {
        if (threadIdx.x == 0) next_problem = atomicAdd(counter, 1ULL);
        __syncthreads();
        const unsigned long long b = next_problem;
        __syncthreads();
        if (b >= (unsigned long long)B) break;
        solve_problem<W, MODEL, PW>(cfg, io, rg, (long)b, smem);
    }
}

// ---- Queue order of mpc_solve_kernel<PW, 1> for large cold-start batches (DESIGN §6, item 3).  From the all-zero start the iteration
// counts spread from ~20 to the 200 cap (p50 42, p99 92 at N = 20), and one iteration costs a warp the same time whether its SM
// is full or not, so a long solve taken late keeps the launch running after the queue is empty.  Taking the problems with the
// longest predicted solve first leaves the short ones to fill the end.  The prediction is a linear score of raw inputs fitted by
// least squares to the oracle's iteration counts (tools/queue_order_model.py: the bench batch to fit, the next 65,536 problems to
// judge; R^2 0.18, but the longest solves come first): the vehicle's distance from the path frame's origin (log), the heading
// change of the reference over the horizon, the previous steering and acceleration commands.  key[b] = the score in 16.16 fixed
// point, clamped to [0, 256): the 24 bits the descending radix sort of (key, index) looks at.
__global__ void __launch_bounds__(256)
queue_key_kernel(const long long B, const int N, const double* state, const double* ref, const double* u_prev, unsigned* key, int* index) {
    const long long nr = 3LL * (N + 1);
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        const double* rp = ref + nr * b + 2 * (N + 1);
        const double s = 69.91 - 5.253 * log1p(hypot(state[4 * b], state[4 * b + 1])) + 0.7904 * fabs(rp[N] - rp[0])
                         + 30.34 * fabs(u_prev[2 * b]) - 1.304 * u_prev[2 * b + 1];
        key[b] = (s > 0.0) ? (unsigned)(fmin(s, 255.99) * 65536.0) : 0u;   // NaN inputs: last
        index[b] = (int)b;
    }
}


// Large batches of the XY model: one THREAD per problem (tpp_solver.cuh).  A lane owns a slot of the state arrays
// ([field][stage][slot]: the 32 lanes of a warp touch 256 contiguous bytes per access) for the whole launch; when its
// problem ends it writes the result and takes the next problem index from the device counter.  The warp leaves when the
// counter has run past the batch and every lane is idle.
#ifndef MPC_TPP_BLOCK
#define MPC_TPP_BLOCK 256
#define MPC_TPP_MIN_BLOCKS 1
#endif
template <int MODEL, int PW = 0>
__global__ void __launch_bounds__(MPC_TPP_BLOCK, MPC_TPP_MIN_BLOCKS)
mpc_solve_tpp_kernel(const KCfg cfg, const BatchPtrs io, const long long B, double* st, double* filt, unsigned long long* counter,
                     const double v_des0) {
    const long slot = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const TppMemT<MODEL> mem(st, filt, cfg.N, slot);
    TppSolverT<MODEL, PW> sv(cfg, mem);
    bool alive = true;   // the counter has not run past the batch for this lane yet
    long b = -1;
    while (__syncthreads_or(alive)) {
        if (alive && b < 0) {
            const unsigned long long nb = atomicAdd(counter, 1ULL);
            if (nb >= (unsigned long long)B) alive = false;
            else if (PW && io.w && !row_weights_ok(io.w, (long)nb, MODEL)) write_error_answer(io, (long)nb);   // the lane takes the next one
            else { b = (long)nb; sv.begin(io, b, v_des0); }
        }
        const bool done = sv.tick(b >= 0);
        if (b >= 0 && done) { sv.finish(io, b); b = -1; }
    }
}

// ---- mpcb200_solve_batch_on_path with the thread-per-problem layout: the waypoints of the whole batch first (warp = problem,
// get_waypoints as in solve_problem), into `ref` = [B][3][N+1] (the caller's ref_out if it asked for one), which the solve kernel
// then reads like references that came from the host; a problem whose path id was never set gets NaN references (its solve ends
// at once) and on_path_invalid_kernel gives it the answer solve_problem gives: MPCB200_ERROR, zero commands.
__global__ void __launch_bounds__(128)
on_path_ref_kernel(const KCfg cfg, const long long B, const double* state, const RefGen rg, double* ref) {
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31, N = cfg.N;
    TeamSolver<1> S(cfg, (smem_t)0);   // (one-warp teams use no shared memory in get_waypoints)
    for (long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < B; b += warps) {
        const int pid = rg.path_of[b];
        double xr = __longlong_as_double(0x7ff8000000000000LL), yr = xr, pr = xr;
        bool sc = false;
        if (!(pid < 0 || pid > 2 || rg.paths[pid].n < 2))
            sc = S.get_waypoints(rg.paths[pid], cfg.dt, state[4 * b], state[4 * b + 1], state[4 * b + 2], !rg.track_using_time, rg.target_vel, xr, yr, pr);
        if (lane <= N) { double* ro = ref + 3LL * (N + 1) * b; ro[lane] = xr; ro[(N + 1) + lane] = yr; ro[2 * (N + 1) + lane] = pr; }
        if (rg.stop && lane == 0) rg.stop[b] = sc ? 1 : 0;
        __syncwarp();
    }
}

__global__ void __launch_bounds__(128)
on_path_invalid_kernel(const long long B, const RefGen rg, const BatchPtrs io) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int pid = rg.path_of[b];
    if (!(pid < 0 || pid > 2 || rg.paths[pid].n < 2)) return;
    write_error_answer(io, b);
}

// ---- Closed-loop fleets with the thread-per-problem layout: one control period = three launches over the whole fleet
// instead of one persistent kernel that carries four vehicles per block through all their periods.
//   plant      thread = vehicle: the ten 100 Hz publishes of ten Euler sub-steps (vehicle_simulator.py:58-112): every lane of a
//              warp integrates its own vehicle (in mpc_rollout_kernel one warp per block does it for four while three wait)
//   waypoints  warp = vehicle: get_waypoints (ref_gps_traj.py:131-218) written straight into the vehicle's slot of the solver state
//   solve      thread = vehicle: the slot still holds the previous solution = the warm start (mpc_cmd_pub.jl:115-141), all
//              vehicles start together and take about the same handful of iterations, which is where this layout is at its best
// Vehicle state is structure-of-arrays [12][Bp]: X Y psi vx vy wz acc df | acc_des df_des | d_f_current acc_current.
#define RV_NF 12
__global__ void __launch_bounds__(128)
rollout_plant_kernel(const long long B, const long long Bp, double* veh, const double* pose0, const int first) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= B) return;
    double st[8], ad, dd;
    if (first) {
        st[0] = pose0[3 * v]; st[1] = pose0[3 * v + 1]; st[2] = pose0[3 * v + 2];
        for (int i = 3; i < 8; i++) st[i] = 0.0;
        ad = 0.0; dd = 0.0;
        veh[8 * Bp + v] = 0.0; veh[9 * Bp + v] = 0.0; veh[10 * Bp + v] = 0.0; veh[11 * Bp + v] = 0.0;
    } else {
        for (int i = 0; i < 8; i++) st[i] = veh[i * Bp + v];
        ad = veh[8 * Bp + v]; dd = veh[9 * Bp + v];
    }
    MPC_NOUNROLL for (int i = 0; i < 10; i++) plant_step(st, ad, dd);
    for (int i = 0; i < 8; i++) veh[i * Bp + v] = st[i];
}

__global__ void __launch_bounds__(128)
rollout_waypoints_kernel(const KCfg cfg, const long long B, const long long Bp, const double* veh, const int* path_of, const RefGen rg,
                         double* tpp_state, double* tpp_filt, int* stop, const int first) {
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    TeamSolver<1> S(cfg, (smem_t)0);   // (one-warp teams use no shared memory in get_waypoints)
    for (long long v = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < B; v += warps) {
        if (first && lane == 0) stop[v] = 0;
        if (!first && stop[v]) continue;   // the stop latch (mpc_cmd_pub.jl:102-111): no more solves, no more references
        double xr, yr, pr;
        const bool sc = S.get_waypoints(rg.paths[path_of[v]], cfg.dt, veh[v], veh[Bp + v], veh[2 * Bp + v], !rg.track_using_time, rg.target_vel, xr, yr, pr);
        if (lane <= cfg.N) {
            const TppMem mem(tpp_state, tpp_filt, cfg.N, (long)v);
            mem.sto(TF_XR, lane, xr); mem.sto(TF_YR, lane, yr); mem.sto(TF_PR, lane, pr);
        }
        if (sc && lane == 0) stop[v] = 1;
        __syncwarp();
    }
}

// MODEL 0: reference samples already in the slots, stop latch, the first solve from the module-load solution `warm0`.
// MODEL 1 (closed loop of the Frenet node, gazebo_sim_mpc_cmd_pub_frenet.jl:112-153): `fref` = [6][Bp] curvature polynomial (4),
// e_y, psi_start per vehicle from rollout_frenet_ref_kernel; state (0, e_y, -psi_start, v); the first solve from all zeros.
// PW: each vehicle's cost weights from out.w (mpcb200_rollout_w, mpcb200_rollout_frenet_w), the slot keeps its vehicle and so its row
template <int MODEL, int PW = 0>
__global__ void __launch_bounds__(MPC_TPP_BLOCK, MPC_TPP_MIN_BLOCKS)
rollout_solve_tpp_kernel(const KCfg cfg, const long long B, const long long Bp, double* veh, const int* stop, double* tpp_state, double* tpp_filt,
                         const double* warm0, const double des_speed, BatchPtrs out, double* log_row, const double* fref, const int first) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = v < B;
    const TppMemT<MODEL> mem(tpp_state, tpp_filt, cfg.N, (long)(valid ? v : 0));
    TppSolverT<MODEL, PW> sv(cfg, mem);
    if (PW && valid && out.w) sv.wr = out.w + (MODEL ? 7 : 8) * v;
    const bool stopped = valid && !MODEL && stop[v] != 0;
    bool live = valid && !stopped;
    double st4[4] = {0.0, 0.0, 0.0, 0.0};
    if (valid) for (int i = 0; i < 4; i++) st4[i] = veh[i * Bp + v];
    if (live) {
        if (MODEL) {
            for (int i = 0; i < 4; i++) sv.kp[i] = fref[i * Bp + v];
            const double c7[7] = {0.0, fref[4 * Bp + v], -fref[5 * Bp + v], st4[3], veh[10 * Bp + v], veh[11 * Bp + v], des_speed};
            if (first) {   // start = 0.0, then the previous solution
                for (int k = 0; k <= cfg.N; k++) for (int f = TF_SX; f <= TF_UD; f++) mem.sto(f, k, 0.0);
                for (int k = 0; k <= cfg.N; k++) { mem.sto(TF_XR, k, 0.0); mem.sto(TF_YR, k, 0.0); mem.sto(TF_PR, k, 0.0); }
            }
            sv.begin_in_place(c7, nullptr);
        } else {
            const double c7[7] = {st4[0], st4[1], st4[2], st4[3], veh[10 * Bp + v], veh[11 * Bp + v], des_speed};
            sv.begin_in_place(c7, warm0);
        }
    }
    bool solved = false;
    while (__syncthreads_or(live)) {
        const bool done = sv.tick(live);
        if (live && done) { sv.finish(out, (long)v); live = false; solved = true; }
    }
    if (!valid) return;
    double acc_des = -1.0, df_des = 0.0, status = -1.0, iters = 0.0;   // stopped: mpc_cmd_pub.jl:148-153
    if (solved) {
        acc_des = out.u0[2 * v]; df_des = out.u0[2 * v + 1]; status = (double)out.status[v]; iters = (double)out.iters[v];
        veh[10 * Bp + v] = df_des; veh[11 * Bp + v] = acc_des;   // update_current_input(df_opt, a_opt) (:140)
    }
    veh[8 * Bp + v] = acc_des; veh[9 * Bp + v] = df_des;         // published whatever the status (:129-132)
    if (log_row) {
        double* r = log_row + 8 * v;
        r[0] = st4[0]; r[1] = st4[1]; r[2] = st4[2]; r[3] = st4[3]; r[4] = acc_des; r[5] = df_des; r[6] = status; r[7] = iters;
    }
}

// Frenet node, per control period and vehicle (warp = vehicle): frenet_reference (mpc_kernel.cuh; nav_msgs_path_frenet.py:44-86) ->
// curvature polynomial, e_y, psi_start, kept per vehicle for the solve kernel
__global__ void __launch_bounds__(128)
rollout_frenet_ref_kernel(const KCfg cfg, const FrenetRolloutArgs a, const long long Bp, const double* veh, double* fref) {
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int k = threadIdx.x & 31;
    TeamSolver<1, 1> S(cfg, (smem_t)0);   // (one-warp teams: collectives are shuffles only)
    for (long long v = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < a.B; v += warps) {
        double kc[4], ey, psi0;
        frenet_reference(S, a.paths[a.path_of[v]], a, veh[v], veh[Bp + v], veh[2 * Bp + v], kc, ey, psi0);
        if (k < 6) fref[k * Bp + v] = (k < 4) ? sel8(kc, k) : (k == 4 ? ey : psi0);
        __syncwarp();
    }
}

// ---- mpcb200_solve_batch_frenet_on_path: the reference of every problem first (warp = problem, frenet_on_path_problem: the
// node's reference step from the pose) into k_out / state_out = [B][4]; the solve kernels then read those rows as an ordinary
// Frenet batch (launch_solve), so the results are those of mpcb200_solve_batch_frenet on the returned inputs by construction.
// vdes_out [B] or null: target_vel for every problem when the caller gives no v_des.  The reference is not fused into the solve
// kernels: that would be a new build of every (WPB, PW) and long-team solve instantiation (DESIGN §3.4).
__global__ void __launch_bounds__(128)
on_path_frenet_ref_kernel(const KCfg cfg, const FrenetRolloutArgs a, const double* pose, double* k_out, double* state_out,
                          double* vdes_out, const double target_vel) {
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    TeamSolver<1, 1> S(cfg, (smem_t)0);   // (one-warp teams: collectives are shuffles only)
    for (long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < a.B; b += warps) {
        frenet_on_path_problem(S, a, pose, (long)b, k_out, state_out);
        if (vdes_out && (threadIdx.x & 31) == 0) vdes_out[b] = target_vel;
        __syncwarp();
    }
}

__global__ void rollout_final_kernel(const long long B, const long long Bp, const double* veh, double* final_state) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= B) return;
    for (int i = 0; i < 8; i++) final_state[8 * v + i] = veh[i * Bp + v];
}

// Tracking metrics of the per-period pipeline (mpcb200_rollout_metrics / _frenet_metrics), launched after the solve of period t:
// warp = vehicle, metrics_period on the pose in veh (which the solve does not move), the published command veh[8..9], and the
// solve's status and iterations unless the stop latch (XY: stop[v]; Frenet: stop = null) kept the vehicle from solving.  The
// waypoint and reference kernels stay as they are, so the nearest sample is searched a second time here.
__global__ void __launch_bounds__(128)
rollout_metrics_kernel(const KCfg cfg, const RolloutArgs a, const long long Bp, const double* veh, const int* stop, const int* status,
                       const int* iters, const int t) {
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    TeamSolver<1> S(cfg, (smem_t)0);   // (one-warp teams use no shared memory in nearest_sample)
    for (long long v = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < a.B; v += warps) {
        const bool solved = !stop || !stop[v];
        metrics_period(S, a.met + v, Bp, t, a.paths[a.path_of[v]], veh[v], veh[Bp + v], veh[2 * Bp + v], veh[8 * Bp + v], veh[9 * Bp + v],
                       solved ? status[v] : -1, solved ? iters[v] : 0);
        __syncwarp();
    }
}

// [B][MET_FIELDS] rows from the [MET_K][stride] accumulators (both the fused kernels and the pipeline)
__global__ void rollout_metrics_final_kernel(const long long B, const long long stride, const double* met, double* out) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= B) return;
    metrics_finalize(met + v, (long)stride, out + (long long)MET_FIELDS * v);
}

#ifndef MPC_ROLLOUT_MIN_BLOCKS
#define MPC_ROLLOUT_MIN_BLOCKS 3
#endif
// PW (this kernel and mpc_rollout_long_kernel): each vehicle's cost weights from args.w (mpcb200_rollout_w)
// MET (these two and mpc_rollout_frenet_kernel): 1 = tracking metrics into args.met (mpcb200_rollout_metrics); a compile-time switch
// like PW, so that the MET = 0 instantiations are the code they always were
template <int PW, int MET = 0>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, MPC_ROLLOUT_MIN_BLOCKS)
mpc_rollout_kernel(const KCfg cfg, const RolloutArgs args, unsigned long long* counter) {
    extern __shared__ double smem_all[];
    const int warp = threadIdx.x >> 5;
    const smem_t smem = smem_base(smem_all + (size_t)warp * smem_doubles_per_team(cfg.N, 0, PW));
    const smem_t px = smem_base(smem_all + (size_t)WARPS_PER_BLOCK * smem_doubles_per_team(cfg.N, 0, PW));   // plant exchange area
    __shared__ unsigned long long next_group;
    TeamSolver<1>::init_work(smem, cfg.N);
    for (;;) {   // the block takes WARPS_PER_BLOCK vehicles at a time and steps them together
        if (threadIdx.x == 0) next_group = atomicAdd(counter, (unsigned long long)WARPS_PER_BLOCK);
        __syncthreads();
        const unsigned long long b0 = next_group;
        __syncthreads();
        if (b0 >= (unsigned long long)args.B) break;
        rollout_group<1, PW, MET>(cfg, args, (long)b0, smem, px, WARPS_PER_BLOCK);
    }
}

// Closed-loop rollouts at long horizons (32 <= N <= 95): one vehicle per block of W = 2 or 3 warps
template <int W, int PW = 0, int MET = 0>
__global__ void __launch_bounds__(W * 32, W == 2 ? 4 : 2)
mpc_rollout_long_kernel(const KCfg cfg, const RolloutArgs args, unsigned long long* counter) {
    extern __shared__ double smem_all[];
    __shared__ unsigned long long next_vehicle;
    const smem_t smem = smem_base(smem_all);
    const smem_t px = smem_base(smem_all + (size_t)smem_doubles_per_team(cfg.N, 0, PW));
    TeamSolver<W>::init_work(smem, cfg.N);
    for (;;) {
        if (threadIdx.x == 0) next_vehicle = atomicAdd(counter, 1ULL);
        __syncthreads();
        const unsigned long long b0 = next_vehicle;
        __syncthreads();
        if (b0 >= (unsigned long long)args.B) break;
        rollout_group<W, PW, MET>(cfg, args, (long)b0, smem, px, 1);
    }
}

// Closed loop on the Frenet-frame module (gazebo_sim_mpc_cmd_pub_frenet.jl:112-153): four vehicles per block
// met: [MET_K][B] accumulators of MET = 1 (rollout_group_frenet)
// PW: each vehicle's cost weights from w = [B][7] (mpcb200_rollout_frenet_w); an argument after met so that the PW = 0 kernels keep theirs
template <int MET = 0, int PW = 0>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, 2)
mpc_rollout_frenet_kernel(const KCfg cfg, const FrenetRolloutArgs args, unsigned long long* counter, double* met, const double* w) {
    extern __shared__ double smem_all[];
    const int warp = threadIdx.x >> 5;
    const smem_t smem = smem_base(smem_all + (size_t)warp * smem_doubles_per_team(cfg.N, 1, PW));
    const smem_t px = smem_base(smem_all + (size_t)WARPS_PER_BLOCK * smem_doubles_per_team(cfg.N, 1, PW));
    __shared__ unsigned long long next_group;
    TeamSolver<1, 1>::init_work(smem, cfg.N);
    for (;;) {
        if (threadIdx.x == 0) next_group = atomicAdd(counter, (unsigned long long)WARPS_PER_BLOCK);
        __syncthreads();
        const unsigned long long b0 = next_group;
        __syncthreads();
        if (b0 >= (unsigned long long)args.B) break;
        rollout_group_frenet<MET, PW>(cfg, args, (long)b0, smem, px, WARPS_PER_BLOCK, met, w);
    }
}

// FP64 FMA throughput probe: 8 independent chains per thread
__global__ void fp64_peak_kernel(double* out, int iters) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 0.999999, c = 1e-9;
    for (int i = 0; i < iters; i++) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

}  // namespace

struct mpcb200_handle {
    mpcb200_config cfg;
    double w[8];
    int device = 0;
    int num_sms = 0;
    int blocks_per_sm = 0;
    int team_warps = 1;     /* warps per problem: 1 (N <= 31), 2 (N <= 63), 3 (N <= 95) */
    int model = 0;          /* 0: XY model; 1: Frenet-frame variant (mpcb200_create_frenet) */
    int frenet_wpb = WARPS_PER_BLOCK;   /* warps (= problems) per block of mpc_solve_frenet_kernel */
    size_t smem_bytes = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    unsigned long long* d_counter = nullptr;
    int* d_roles = nullptr;   /* lane roles of the Riccati recursion for this horizon (riccati_roles) */
    DevBuf d_state, d_ref, d_vdes, d_uprev, d_warm, d_u0, d_cost, d_status, d_iters, d_traj;
    DevBuf d_path[3], d_pose, d_pathof, d_log, d_final, d_stop;
    DevBuf d_tpp_state, d_tpp_filt;   /* thread-per-problem path: slot state [warp][stage][field][lane], filters */
    DevBuf d_genref;                  /* ... on a path: the generated waypoints [B][3][N+1] when the caller did not ask for them */
    DevBuf d_veh, d_vstop;            /* ... closed-loop fleets: vehicle state [12][Bp], stop latches */
    DevBuf d_w;                       /* per-problem weight rows of a weighted call (host pointers) */
    DevBuf d_met, d_metout;           /* rollout tracking metrics: accumulators [MET_K][stride], rows [B][MET_FIELDS] */
    DevBuf d_order;                   /* queue order of large cold-start batches: keys, indices (in, out) and the sort's scratch */
    int64_t order_min_batch = 1;      /* ... taken from this many problems on */
    int blocks_per_sm_ord = 0;        /* resident blocks per SM of the queue-ordered one-warp XY solve kernel (mpc_solve_kernel<0, 1>) */
    int blocks_per_sm_w = 0;          /* resident blocks per SM of the PW = 1 solve kernel of this handle (8 more doubles per team) */
    int rollout_blocks_per_sm_w = 0;  /* ... of the PW = 1 fused rollout kernel */
    int tpp_blocks_per_sm = 0;        /* resident blocks of mpc_solve_tpp_kernel per SM */
    int tpp_block = MPC_TPP_BLOCK;    /* threads per block of mpc_solve_tpp_kernel (a multiple of 32, <= MPC_TPP_BLOCK) */
    bool tpp_block_forced = false;    /* ... given by MPCB200_TPP_BLOCK: no per-batch choice */
    int64_t tpp_min_batch = 0;        /* batches of at least this many problems take the thread-per-problem path (0: never) */
    bool tpp_default_rule = true;     /* ... as set by the default rule (then warm / rollout starts switch at half of it) */
    DevBuf d_rec, d_resto;        /* packed 32-byte records; restoration count per problem of the last solve */
    DevBuf d_seed;                /* the module-load solution (start point of a rollout's first solve), [6N+4] */
    DevBuf d_fit;                 /* Frenet rollouts: the two least-squares fit matrices [4][n1], [4][n2] */
    double fit_window = -1.0;     /* ... built for this window length */
    int fit_n1 = 0, fit_n2 = 0;
    int frenet_rollout_blocks_per_sm = 0;
    bool seed_valid = false;
    int64_t last_B = 0;           /* batch of the last solve (mpcb200_get_restorations) */
    int32_t small_resto[64];      /* ... its restoration counts when it went through the small-batch path */
    bool resto_on_host = false;
    /* multi-GPU: the handle itself works on devices[0]; sub[i] on devices[i + 1] */
    int n_sub = 0;
    mpcb200_handle* sub[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int64_t slice_lo[8] = {0, 0, 0, 0, 0, 0, 0, 0}, slice_hi[8] = {0, 0, 0, 0, 0, 0, 0, 0};   /* slices of the last sharded call */
    bool last_sharded = false;
    DevBuf d_stage;               /* small batches: one contiguous device buffer, one copy each way */
    void* h_stage = nullptr;      /* its pinned host mirror */
    size_t h_stage_cap = 0;
    /* small batches on the handle's own stream: copy in -> kernel -> copy out captured once per shape as a CUDA graph
     * (one cudaGraphLaunch instead of five driver calls per solve); dropped when a buffer, the handle's weights or the stream
     * change.  A shape is B and which optional buffers the call has, per-problem weight rows included */
    struct SmallGraph { int64_t B; int flags; cudaGraphExec_t exec; };
    SmallGraph graphs[8];
    int n_graphs = 0;
    bool graphs_ok = true;
    int path_n[3] = {0, 0, 0};
    int rollout_blocks_per_sm = 0;
    mpcb200_stats stats;
    char err[512];
};

static thread_local char g_err[512] = "";

/* The dynamic shared-memory limit of a kernel is an attribute of the FUNCTION (per device), not of a launch, and the team
 * footprint depends on the horizon: handles with different horizons in one process share it.  It is therefore only ever
 * raised (a larger limit is fine for a smaller launch); lowering it made the next launch of a longer-horizon handle fail
 * with "invalid argument". */
static cudaError_t raise_dyn_smem(const void* fn, int device, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> current;
    std::lock_guard<std::mutex> g(mu);
    size_t& cur = current[std::make_pair(fn, device)];
    if (cur >= bytes) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) cur = bytes;
    return e;
}

static int fail(mpcb200_handle* h, int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    char* dst = h ? h->err : g_err;
    vsnprintf(dst, 512, fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(h, expr)                                                                          \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess) return fail(h, MPCB200_ECUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

static void drop_graphs(mpcb200_handle* h) {
    for (int i = 0; i < h->n_graphs; i++) if (h->graphs[i].exec) cudaGraphExecDestroy(h->graphs[i].exec);
    h->n_graphs = 0;
}

static int ensure(mpcb200_handle* h, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap) return 0;
    if (b.p) CUDA_TRY(h, cudaFree(b.p));
    b.p = nullptr; b.cap = 0;
    size_t cap = bytes + bytes / 4;
    CUDA_TRY(h, cudaMalloc(&b.p, cap));
    b.cap = cap;
    return 0;
}

static KCfg make_kcfg(const mpcb200_handle* h) {
    KCfg k;
    memset(&k, 0, sizeof(k));
    const mpcb200_config& c = h->cfg;
    k.N = c.N; k.max_iter = c.max_iter; k.start_mode = c.start_mode;
    k.dt = c.dt; k.dtc = c.dt_control; k.La = c.L_a; k.Lb = c.L_b;
    k.vmin = c.v_min; k.vmax = c.v_max; k.amax = c.a_max; k.smax = c.steer_max;
    k.admax = c.a_dmax; k.sdmax = c.steer_dmax; k.tol = c.tol;
    for (int i = 0; i < 8; i++) k.w[i] = h->w[i];
    kcfg_finalize(k);
    k.roles = h->d_roles;
    return k;
}

/* problems per block of the warp / block-per-problem solve kernel */
static int teams_per_block(const mpcb200_handle* h) { return (h->team_warps != 1) ? 1 : (h->model ? h->frenet_wpb : WARPS_PER_BLOCK); }

/* the warp / block-per-problem solve kernel of a handle (model, team size, Frenet block size) and its threads per block */
typedef void (*TeamKernel)(const KCfg, const BatchPtrs, const RefGen, const long long, unsigned long long*, const int*);
template <int PW>
static TeamKernel team_kernel(const mpcb200_handle* h, int* threads) {
    *threads = 32 * h->team_warps;
    if (h->model && h->team_warps == 2) return mpc_solve_long_kernel<2, 1, PW>;
    if (h->model && h->team_warps == 3) return mpc_solve_long_kernel<3, 1, PW>;
    if (h->model) { *threads = 32 * h->frenet_wpb; return (h->frenet_wpb == 3) ? mpc_solve_frenet_kernel<3, PW> : mpc_solve_frenet_kernel<4, PW>; }
    if (h->team_warps == 1) { *threads = 32 * WARPS_PER_BLOCK; return mpc_solve_kernel<PW>; }
    return (h->team_warps == 2) ? mpc_solve_long_kernel<2, 0, PW> : mpc_solve_long_kernel<3, 0, PW>;
}

/* the fused closed-loop kernel of an XY handle */
typedef void (*RolloutKernel)(const KCfg, const RolloutArgs, unsigned long long*);
template <int PW, int MET = 0>
static RolloutKernel rollout_kernel(const mpcb200_handle* h) {
    if (h->team_warps == 1) return mpc_rollout_kernel<PW, MET>;
    return (h->team_warps == 2) ? mpc_rollout_long_kernel<2, PW, MET> : mpc_rollout_long_kernel<3, PW, MET>;
}

/* dynamic shared memory of the fused rollout kernel: the teams and the plant exchange area (the XY handle's smem_bytes already
 * holds it at N <= 31; the Frenet kernel always runs WARPS_PER_BLOCK vehicles per block, whatever frenet_wpb is) */
static size_t rollout_smem_bytes(const mpcb200_handle* h, bool pw) {
    if (h->model) return WARPS_PER_BLOCK * ((size_t)smem_doubles_per_team(h->cfg.N, 1, pw) + ROLLOUT_PX) * sizeof(double);
    return h->smem_bytes + (h->team_warps == 1 ? 0 : ROLLOUT_PX * sizeof(double)) + (pw ? (size_t)teams_per_block(h) * 8 * sizeof(double) : 0);
}

/* shared-memory limit, carveout and resident blocks per SM of one kernel */
static cudaError_t prepare_kernel(const void* fn, int device, int threads, size_t bytes, int* blocks_per_sm) {
    cudaError_t e = raise_dyn_smem(fn, device, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, fn, threads, bytes);
    if (*blocks_per_sm < 1) *blocks_per_sm = 1;
    return e;
}

extern "C" {

int mpcb200_version(void) { return MPCB200_VERSION; }

int mpcb200_default_config(mpcb200_config* c, int32_t N) {
    if (!c) return MPCB200_EINVAL;
    memset(c, 0, sizeof(*c));
    c->N = N;
    c->max_iter = 200;
    c->start_mode = MPCB200_START_ZERO;
    c->device = 0;
    c->dt = 0.20;          /* MKZMPCPathFollower.jl:33 */
    c->dt_control = 0.10;  /* :28 */
    c->L_a = 1.108;        /* :31 */
    c->L_b = 1.742;        /* :32 */
    c->v_min = 0.0;        /* :47 */
    c->v_max = 20.0;       /* :48 */
    c->a_max = 1.0;        /* :44 */
    c->steer_max = 0.5;    /* :41 */
    c->a_dmax = 1.5;       /* :45 */
    c->steer_dmax = 0.5;   /* :42 */
    c->tol = 1e-8;
    c->n_devices = 0;      /* one GPU: `device` */
    return MPCB200_OK;
}

/* The default rule of mpcb200_set_large_batch_path, from measurements on the B200 (profiles/r02_logs/r02_tpp_thresholds.log,
 * r02_tpp_frenet.log).  XY model from the all-zero start: iteration counts spread from 25 to 200, the streaming layout pays for
 * the tail of long solves: N <= 10 only, from 32,768 problems.  Frenet-frame variant: every solve takes 14-17 iterations, the
 * streaming layout wins at every horizon tried (N = 8: 1.3x / 1.9x / 2.1x at 16 K / 64 K / 256 K problems; N = 20: 0.94x / 1.47x /
 * 1.30x at 16 K / 32 K / 64 K; N = 31, 40: 1.29x at 64 K). */
static int64_t tpp_default_min_batch(int model, int N) {
    if (model) return (N <= 10) ? 16384 : 32768;
    return (N <= 10) ? 32768 : 0;
}

/* the module-default weights of MKZMPCPathFollower.jl:51-59 in update_cost order: an XY handle's weights until mpcb200_set_cost,
 * and those of the module-load solve that seeds every rollout */
static const double W_XY_DEFAULT[8] = {9.0, 9.0, 10.0, 0.0, 100.0, 1000.0, 0.0, 0.0};

static int create_impl(mpcb200_handle** out, const mpcb200_config* cfg, int model);
static int create_multi(mpcb200_handle** out, const mpcb200_config* cfg, int model);
int mpcb200_create(mpcb200_handle** out, const mpcb200_config* cfg) { return create_multi(out, cfg, 0); }
int mpcb200_create_frenet(mpcb200_handle** out, const mpcb200_config* cfg) { return create_multi(out, cfg, 1); }

/* n_devices > 1: one full single-GPU handle per device; the first one is the handle the caller holds */
static int create_multi(mpcb200_handle** out, const mpcb200_config* cfg, int model) {
    if (!out || !cfg) return fail(nullptr, MPCB200_EINVAL, "mpcb200_create: NULL argument");
    *out = nullptr;
    if (cfg->n_devices < 0 || cfg->n_devices > 8) return fail(nullptr, MPCB200_EINVAL, "mpcb200_create: n_devices=%d outside [0,8]", cfg->n_devices);
    if (cfg->n_devices <= 1) {
        mpcb200_config c1 = *cfg;
        if (cfg->n_devices == 1) c1.device = cfg->devices[0];
        return create_impl(out, &c1, model);
    }
    for (int i = 0; i < cfg->n_devices; i++)
        for (int j = 0; j < i; j++)
            if (cfg->devices[i] == cfg->devices[j]) return fail(nullptr, MPCB200_EINVAL, "mpcb200_create: device %d listed twice", cfg->devices[i]);
    mpcb200_handle* first = nullptr;
    for (int i = 0; i < cfg->n_devices; i++) {
        mpcb200_config ci = *cfg;
        ci.device = cfg->devices[i];
        mpcb200_handle* hi = nullptr;
        const int rc = create_impl(&hi, &ci, model);
        if (rc) { if (first) mpcb200_destroy(first); return rc; }
        if (i == 0) first = hi; else first->sub[first->n_sub++] = hi;
    }
    first->cfg.n_devices = cfg->n_devices;
    *out = first;
    return MPCB200_OK;
}

static int create_impl(mpcb200_handle** out, const mpcb200_config* cfg, int model) {
    if (!out || !cfg) return fail(nullptr, MPCB200_EINVAL, "mpcb200_create: NULL argument");
    *out = nullptr;
    if (cfg->N < 3 || cfg->N > 95) return fail(nullptr, MPCB200_EINVAL, "mpcb200_create: horizon N=%d outside [3,95]", cfg->N);
    if (cfg->max_iter < 0) return fail(nullptr, MPCB200_EINVAL, "mpcb200_create: max_iter=%d is negative", cfg->max_iter);
    /* every model constant must be finite: an infinite bound or step reaches kcfg_finalize, dtLb and rfrac as inf or NaN */
    const struct { const char* name; double v; bool ok; const char* rule; } consts[] = {
        {"dt", cfg->dt, cfg->dt > 0, "> 0"},
        {"dt_control", cfg->dt_control, cfg->dt_control > 0, "> 0"},
        {"L_a", cfg->L_a, cfg->L_a >= 0, ">= 0"},
        {"L_b", cfg->L_b, cfg->L_b > 0, "> 0"},
        {"v_min", cfg->v_min, true, "< v_max"},
        {"v_max", cfg->v_max, cfg->v_max > cfg->v_min, "> v_min"},
        {"a_max", cfg->a_max, cfg->a_max > 0, "> 0"},
        {"steer_max", cfg->steer_max, cfg->steer_max > 0 && cfg->steer_max < 1.5, "in (0, 1.5)"},
        {"a_dmax", cfg->a_dmax, cfg->a_dmax > 0, "> 0"},
        {"steer_dmax", cfg->steer_dmax, cfg->steer_dmax > 0, "> 0"},
        {"tol", cfg->tol, cfg->tol > 0, "> 0"},
    };
    for (const auto& k : consts)
        if (!k.ok || !std::isfinite(k.v))
            return fail(nullptr, MPCB200_EINVAL, "mpcb200_create: model constant %s = %g must be finite and %s", k.name, k.v, k.rule);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0)
        return fail(nullptr, MPCB200_ENODEVICE, "mpcb200_create: no CUDA device (%s); this library has no CPU path",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, MPCB200_EINVAL, "mpcb200_create: device %d of %d", cfg->device, ndev);
    mpcb200_handle* h = new (std::nothrow) mpcb200_handle();
    if (!h) return fail(nullptr, MPCB200_ENOMEM, "mpcb200_create: out of host memory");
    h->cfg = *cfg;
    h->device = cfg->device;
    h->err[0] = 0;
    memset(&h->stats, 0, sizeof(h->stats));
    /* MKZMPCPathFollowerFrenet.jl:51-58 in the XY slots: nothing on s, C_ey, C_epsi, C_ev, C_dacc, C_ddf, C_acc, C_df */
    const double w1[8] = {0.0, 9.0, 10.0, 0.5, 100.0, 1000.0, 0.0, 0.0};
    memcpy(h->w, model ? w1 : W_XY_DEFAULT, sizeof(w1));
    h->model = model;
#define TRY_OR_FREE(expr)                                                                 \
    do {                                                                                  \
        cudaError_t e2 = (expr);                                                          \
        if (e2 != cudaSuccess) {                                                          \
            fail(nullptr, MPCB200_ECUDA, "%s: %s", #expr, cudaGetErrorString(e2));        \
            mpcb200_destroy(h);   /* releases whatever was created so far */              \
            return MPCB200_ECUDA;                                                         \
        }                                                                                 \
    } while (0)
    TRY_OR_FREE(cudaSetDevice(h->device));
    cudaDeviceProp prop;
    TRY_OR_FREE(cudaGetDeviceProperties(&prop, h->device));
    h->num_sms = prop.multiProcessorCount;
    TRY_OR_FREE(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    TRY_OR_FREE(cudaEventCreate(&h->ev0));
    TRY_OR_FREE(cudaEventCreate(&h->ev1));
    TRY_OR_FREE(cudaMalloc((void**)&h->d_counter, sizeof(unsigned long long)));
    h->team_warps = team_warps(cfg->N);
    {
        int roles[32 * ROLE_STRIDE_F + 32 * RS_STRIDE];   /* shared-memory version, then the register version (MODEL 0) */
        const int rs = role_stride_of(model);
        for (int l = 0; l < 32; l++) riccati_roles(l, cfg->N, w_sd_of(h->team_warps, model), roles + l * rs, model);
        for (int l = 0; l < 32; l++) riccati_roles_shfl(l, cfg->N, w_sd_of(h->team_warps, model), roles + 32 * rs + l * RS_STRIDE);
        TRY_OR_FREE(cudaMalloc((void**)&h->d_roles, sizeof(roles)));
        TRY_OR_FREE(cudaMemcpy(h->d_roles, roles, sizeof(int) * (32 * rs + 32 * RS_STRIDE), cudaMemcpyHostToDevice));
    }
    const size_t team = (size_t)smem_doubles_per_team(cfg->N, model) * sizeof(double);
    if (model && h->team_warps == 1) {
        int b4 = 0, b3 = 0;
        TRY_OR_FREE(prepare_kernel((const void*)mpc_solve_frenet_kernel<4>, h->device, 4 * 32, 4 * team, &b4));
        TRY_OR_FREE(prepare_kernel((const void*)mpc_solve_frenet_kernel<3>, h->device, 3 * 32, 3 * team, &b3));
        /* measured (tools/frenet_bench.py): N = 8: 12 warps at 168 registers 6.06 M solves/s vs 8 warps at 255 registers 5.80 M;
         * N = 20: 9 warps 2.88 M vs 8 warps 3.23 M -- the spill code of the 168-register build pays only for >= 1.4x the warps */
        h->frenet_wpb = (10 * 3 * b3 >= 14 * 4 * b4) ? 3 : 4;
        if (const char* e = getenv("MPCB200_FRENET_WPB")) { int v = atoi(e); if (v == 3 || v == 4) h->frenet_wpb = v; }  /* tuning aid */
        h->blocks_per_sm = (h->frenet_wpb == 3) ? b3 : b4;
        h->smem_bytes = h->frenet_wpb * team;
        TRY_OR_FREE(prepare_kernel((const void*)mpc_rollout_frenet_kernel<0>, h->device, WARPS_PER_BLOCK * 32, rollout_smem_bytes(h, false),
                                   &h->frenet_rollout_blocks_per_sm));
    } else {
        /* one-warp XY teams: four per block, with the plant exchange area of the fused rollout kernel */
        h->smem_bytes = (model || h->team_warps > 1) ? team : WARPS_PER_BLOCK * (team + ROLLOUT_PX * sizeof(double));
        int threads = 0;
        const void* fn = (const void*)team_kernel<0>(h, &threads);
        TRY_OR_FREE(prepare_kernel(fn, h->device, threads, h->smem_bytes, &h->blocks_per_sm));
        if (!model && h->team_warps == 1) {   /* the queue-ordered build of the same kernel (same registers and footprint) */
            TRY_OR_FREE(prepare_kernel((const void*)mpc_solve_kernel<0, 1>, h->device, threads, h->smem_bytes, &h->blocks_per_sm_ord));
        }
        if (!model)
            TRY_OR_FREE(prepare_kernel((const void*)rollout_kernel<0>(h), h->device, threads, rollout_smem_bytes(h, false), &h->rollout_blocks_per_sm));
    }
    {
        /* thread-per-problem path for large batches (any horizon): needs B >> resident lanes to keep them busy */
        const void* tk = model ? (const void*)mpc_solve_tpp_kernel<1> : (const void*)mpc_solve_tpp_kernel<0>;
        TRY_OR_FREE(cudaFuncSetAttribute(tk, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1));
        const void* tkw = model ? (const void*)mpc_solve_tpp_kernel<1, 1> : (const void*)mpc_solve_tpp_kernel<0, 1>;
        TRY_OR_FREE(cudaFuncSetAttribute(tkw, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1));
        TRY_OR_FREE(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->tpp_blocks_per_sm, tk, MPC_TPP_BLOCK, 0));
        if (h->tpp_blocks_per_sm < 1) h->tpp_blocks_per_sm = 1;
        if (const char* e = getenv("MPCB200_TPP_BLOCKS_PER_SM")) { int v = atoi(e); if (v >= 1 && v < h->tpp_blocks_per_sm) h->tpp_blocks_per_sm = v; }  /* tuning aid */
        if (const char* e = getenv("MPCB200_TPP_BLOCK")) { int v = atoi(e); if (v >= 32 && v <= MPC_TPP_BLOCK && v % 32 == 0) { h->tpp_block = v; h->tpp_block_forced = true; } }  /* tuning aid */
        /* measured (tools/tpp_ab.py, profiles/r02_logs/r02_tpp_thresholds.log): N = 8: 0.8x / 1.2x / 1.5x / 1.8x the warp-per-problem
         * kernel at 16 K / 32 K / 64 K / 128 K problems; N = 12, 16: break-even at ~128 K; N = 20: 0.65x at 64 K, 0.97x at 256 K */
        h->tpp_min_batch = tpp_default_min_batch(model, cfg->N);
        if (const char* e = getenv("MPCB200_TPP_MIN_BATCH")) { h->tpp_min_batch = atoll(e); h->tpp_default_rule = false; }   /* tuning aid; 0 switches the path off */
    }
    {
        /* the PW = 1 kernels of the weighted entry points: 8 more doubles of shared memory per team */
        int threads = 0;
        const void* fw = (const void*)team_kernel<1>(h, &threads);
        TRY_OR_FREE(prepare_kernel(fw, h->device, threads, h->smem_bytes + (size_t)teams_per_block(h) * 8 * sizeof(double), &h->blocks_per_sm_w));
        if (!model)
            TRY_OR_FREE(prepare_kernel((const void*)rollout_kernel<1>(h), h->device, threads, rollout_smem_bytes(h, true), &h->rollout_blocks_per_sm_w));
    }
    if (h->blocks_per_sm < 1) h->blocks_per_sm = 1;
    if (const char* e = getenv("MPCB200_BLOCKS_PER_SM")) { int v = atoi(e); if (v >= 1 && v < h->blocks_per_sm) h->blocks_per_sm = v; }  /* tuning aid */
    /* the ordered kernel is the same solver with two more instructions; should it ever fit fewer blocks, its grid follows */
    if (h->blocks_per_sm_ord < 1 || h->blocks_per_sm_ord > h->blocks_per_sm) h->blocks_per_sm_ord = h->blocks_per_sm;
    /* cold-start batches of the one-warp XY kernel take their problems longest predicted solve first (queue_order) from 5/4
     * waves of resident teams on (2,220 problems on a B200).  Measured at N = 20 against counter order, 7 alternated runs
     * (profiles/r05_logs/queue_order_threshold.log; run-to-run spread 1-5 % at these sizes): 1,776 problems (one wave: every
     * problem starts at once, the ~40 us of key kernel and sort are pure cost) +1.3 %, 1,900 +0.6 %, 2,048 -2.8 %, 2,304 -2.8 %,
     * 2,664 -3.2 %, 3,072 -3.2 %, 3,552 -2.2 %; 8,192 -17 %, 65,536 -3.7 % (queue_order_ab.log).  Break-even lies between 1.07
     * and 1.15 waves; the threshold keeps a margin above it for GPUs with other SM counts and for the spread */
    h->order_min_batch = (int64_t)MPC_ORDER_MIN_QUARTER_WAVES * h->num_sms * h->blocks_per_sm_ord * WARPS_PER_BLOCK / 4;
    if (h->order_min_batch < 1) h->order_min_batch = 1;
#undef TRY_OR_FREE
    *out = h;
    return MPCB200_OK;
}

int mpcb200_destroy(mpcb200_handle* h) {
    if (!h) return MPCB200_EINVAL;
    for (int i = 0; i < h->n_sub; i++) if (h->sub[i]) mpcb200_destroy(h->sub[i]);
    h->n_sub = 0;
    cudaSetDevice(h->device);
    DevBuf* bufs[] = {&h->d_state, &h->d_ref, &h->d_vdes, &h->d_uprev, &h->d_warm, &h->d_u0, &h->d_cost, &h->d_status, &h->d_iters, &h->d_traj,
                      &h->d_path[0], &h->d_path[1], &h->d_path[2], &h->d_pose, &h->d_pathof, &h->d_log, &h->d_final, &h->d_stop, &h->d_stage,
                      &h->d_rec, &h->d_resto, &h->d_seed, &h->d_fit, &h->d_tpp_state, &h->d_tpp_filt, &h->d_veh, &h->d_vstop, &h->d_genref,
                      &h->d_w, &h->d_order};
    for (DevBuf* b : bufs) if (b->p) cudaFree(b->p);
    if (h->d_counter) cudaFree(h->d_counter);
    if (h->d_roles) cudaFree(h->d_roles);
    drop_graphs(h);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return MPCB200_OK;
}

int mpcb200_set_cost(mpcb200_handle* h, const double w[8]) {
    if (!h || !w) return fail(h, MPCB200_EINVAL, "mpcb200_set_cost: NULL argument");
    for (int i = 0; i < 8; i++) if (!(w[i] >= 0.0)) return fail(h, MPCB200_EINVAL, "mpcb200_set_cost: weight %d is negative or NaN", i);
    memcpy(h->w, w, 8 * sizeof(double));
    drop_graphs(h);   /* the weights are kernel parameters */
    for (int i = 0; i < h->n_sub; i++) { memcpy(h->sub[i]->w, w, 8 * sizeof(double)); drop_graphs(h->sub[i]); }
    return MPCB200_OK;
}

int mpcb200_set_large_batch_path(mpcb200_handle* h, int64_t min_batch) {
    if (!h) return MPCB200_EINVAL;
    const int64_t v = (min_batch < 0) ? tpp_default_min_batch(h->model, h->cfg.N) : min_batch;
    h->tpp_min_batch = v; h->tpp_default_rule = (min_batch < 0);
    drop_graphs(h);   /* a captured small-batch graph holds the kernel it was captured with */
    for (int i = 0; i < h->n_sub; i++) { h->sub[i]->tpp_min_batch = v; h->sub[i]->tpp_default_rule = (min_batch < 0); drop_graphs(h->sub[i]); }
    return MPCB200_OK;
}

/* the stream of devices[0]; the other devices of a multi-GPU handle keep their own streams */
int mpcb200_set_stream(mpcb200_handle* h, void* s) {
    if (!h) return MPCB200_EINVAL;
    h->stream = s ? (cudaStream_t)s : h->own_stream;
    drop_graphs(h);
    return MPCB200_OK;
}

/* the queue order of mpc_solve_kernel<0, 1>: a key per problem (queue_key_kernel), then a stable descending radix sort of
 * (key, index) over the key's 24 bits; *order = the sorted indices, in h->d_order (sized at the first large batch) */
static int queue_order(mpcb200_handle* h, int64_t B, const BatchPtrs& io, const int** order) {
    const int n = (int)B;
    size_t sort_bytes = 0;
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairsDescending(nullptr, sort_bytes, (const unsigned*)nullptr, (unsigned*)nullptr,
                                                          (const int*)nullptr, (int*)nullptr, n, 0, 24, h->stream));
    const size_t arr = ((size_t)n * sizeof(int) + 255) / 256 * 256;
    int rc;
    if ((rc = ensure(h, h->d_order, 4 * arr + sort_bytes))) return rc;
    char* base = (char*)h->d_order.p;
    unsigned* key_in = (unsigned*)base; unsigned* key_out = (unsigned*)(base + arr);
    int* idx_in = (int*)(base + 2 * arr); int* idx_out = (int*)(base + 3 * arr);
    const long long kb = (B + 255) / 256, kmax = (long long)h->num_sms * 8;
    queue_key_kernel<<<(int)(kb < kmax ? kb : kmax), 256, 0, h->stream>>>((long long)B, h->cfg.N, io.state, io.ref, io.u_prev, key_in, idx_in);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairsDescending(base + 4 * arr, sort_bytes, key_in, key_out, idx_in, idx_out, n, 0, 24, h->stream));
    h->stats.kernel_launches += 2;   /* the key kernel and the sort (one call of cub's radix sort, which launches several kernels) */
    *order = idx_out;
    return 0;
}

static int launch_solve(mpcb200_handle* h, int64_t B, const BatchPtrs& io, const RefGen& rg, unsigned long long* zeroed_counter = nullptr) {
    unsigned long long* counter = zeroed_counter ? zeroed_counter : h->d_counter;
    if (!zeroed_counter) CUDA_TRY(h, cudaMemsetAsync(h->d_counter, 0, sizeof(unsigned long long), h->stream));
    /* (never for the packed small-batch path, which brings its own counter and may be inside a graph capture) */
    /* starts next to the solution (warm start, rollout start) take a handful of iterations each, all about the same number:
     * no tail of long solves, so the streaming layout already pays at half the batch (measured at N = 8, 16,384 problems:
     * 1.06x warm, 1.30x from the rollout start; profiles/r02_logs/r02_tpp_warm.log) */
    const int64_t tpp_from = (h->tpp_default_rule && !h->model && (io.warm || h->cfg.start_mode == MPCB200_START_ROLLOUT)) ? h->tpp_min_batch / 2 : h->tpp_min_batch;
    const bool tpp_path_ok = !rg.path_of || (!h->model && h->team_warps == 1);   /* waypoints by one-warp teams: N <= 31 */
    if (tpp_path_ok && !zeroed_counter && h->tpp_min_batch > 0 && B >= tpp_from) {
        /* thread-per-problem: as many slots as lanes can be resident, never more than problems.  The block size is the one that
         * fills the last wave best: when every solve takes about the same number of trips (Frenet variant, warm starts) a batch of
         * 1.73 x the resident lanes leaves a quarter of them idle for the second half of the launch (Frenet N = 20, 65,536
         * problems: 14.2 ms with 224-thread blocks = 1.98 waves, 15.5 ms with 256) */
        int tb = h->tpp_block;
        if (!h->tpp_block_forced) {
            long long best = -1;
            for (int cand = MPC_TPP_BLOCK; cand >= MPC_TPP_BLOCK - 96; cand -= 32) {
                const long long per_wave = (long long)h->num_sms * h->tpp_blocks_per_sm * cand;
                const long long cost = ((B + per_wave - 1) / per_wave) * cand;     /* lane-slots reserved per SM over the launch */
                if (best < 0 || cost < best) { best = cost; tb = cand; }
            }
        }
        long long blocks = (long long)h->num_sms * h->tpp_blocks_per_sm;
        const long long need = (B + tb - 1) / tb;
        if (blocks > need) blocks = need;
        const long long S = blocks * tb;
        int rc;
        if ((rc = ensure(h, h->d_tpp_state, tpp_state_doubles(h->cfg.N, (long)S, h->model) * sizeof(double)))) return rc;
        if ((rc = ensure(h, h->d_tpp_filt, tpp_filter_doubles((long)S) * sizeof(double)))) return rc;
        BatchPtrs io2 = io;
        if (rg.path_of) {
            double* ref = rg.ref_out;
            if (!ref) {
                if ((rc = ensure(h, h->d_genref, (size_t)B * 3 * ((size_t)h->cfg.N + 1) * sizeof(double)))) return rc;
                ref = (double*)h->d_genref.p;
            }
            const long long wblocks = (B + 3) / 4, wmax = (long long)h->num_sms * 16;
            on_path_ref_kernel<<<(int)(wblocks < wmax ? wblocks : wmax), 128, 0, h->stream>>>(make_kcfg(h), (long long)B, io.state, rg, ref);
            CUDA_TRY(h, cudaGetLastError());
            io2.ref = ref;
            h->stats.kernel_launches += 1;
        }
        const double v_des0 = rg.path_of ? rg.target_vel : 0.0;   /* des_speed when the caller gives no v_des, mpc_cmd_pub.jl:58-62,116 */
        auto tk = h->model ? (io.w ? mpc_solve_tpp_kernel<1, 1> : mpc_solve_tpp_kernel<1, 0>) : (io.w ? mpc_solve_tpp_kernel<0, 1> : mpc_solve_tpp_kernel<0, 0>);
        tk<<<(int)blocks, tb, 0, h->stream>>>(make_kcfg(h), io2, (long long)B, (double*)h->d_tpp_state.p, (double*)h->d_tpp_filt.p, counter, v_des0);
        CUDA_TRY(h, cudaGetLastError());
        h->stats.kernel_launches += 1;
        if (rg.path_of) {
            on_path_invalid_kernel<<<(int)((B + 127) / 128), 128, 0, h->stream>>>((long long)B, rg, io);
            CUDA_TRY(h, cudaGetLastError());
            h->stats.kernel_launches += 1;
        }
        return 0;
    }
    const int tpb = teams_per_block(h);
    const bool pw = io.w != nullptr;
    /* longest predicted solve first (queue_key_kernel): XY one-warp teams, references from the caller, cold starts with the
     * handle's weights -- what the score was fitted on; warm and rollout starts take a few iterations each, no tail to cut */
    const bool ordered = B >= h->order_min_batch && B <= INT32_MAX && !zeroed_counter && !h->model && h->team_warps == 1 &&
                         !rg.path_of && !io.warm && !pw && h->cfg.start_mode == MPCB200_START_ZERO;
    long long blocks_needed = (B + tpb - 1) / tpb;
    long long max_blocks = (long long)h->num_sms * (pw ? h->blocks_per_sm_w : (ordered ? h->blocks_per_sm_ord : h->blocks_per_sm));
    int grid = (int)(blocks_needed < max_blocks ? blocks_needed : max_blocks);
    if (grid < 1) grid = 1;
    int threads = 0;
    TeamKernel tk = pw ? team_kernel<1>(h, &threads) : team_kernel<0>(h, &threads);
    const size_t smem = h->smem_bytes + (pw ? (size_t)tpb * 8 * sizeof(double) : 0);
    const int* order = nullptr;
    if (ordered) {
        int rc;
        if ((rc = queue_order(h, B, io, &order))) return rc;
        tk = mpc_solve_kernel<0, 1>;
    }
    tk<<<grid, threads, smem, h->stream>>>(make_kcfg(h), io, rg, (long long)B, counter, order);
    CUDA_TRY(h, cudaGetLastError());
    h->stats.kernel_launches += 1;
    return 0;
}

static void fill_paths(const mpcb200_handle* h, PathTable* paths) {
    for (int i = 0; i < 3; i++) {
        const double* base = (const double*)h->d_path[i].p;
        const int n = h->path_n[i];
        memset(&paths[i], 0, sizeof(PathTable));
        paths[i].n = n;
        if (n) { paths[i].t = base; paths[i].X = base + n; paths[i].Y = base + 2 * (size_t)n; paths[i].psi = base + 3 * (size_t)n; paths[i].s = base + 4 * (size_t)n;
                 paths[i].cb = base + 5 * (size_t)n; paths[i].nch = path_chunks(n); }
    }
}

/* the arguments of one solve call (host or device pointers) */
struct SolveArgs {
    const char* who;
    const double* state; const double* ref; const int32_t* path_of;
    int32_t track_using_time; double target_vel;
    const double* v_des; const double* u_prev; double* warm;
    double* u0; double* cost; int32_t* status; int32_t* iters; double* traj;
    double* ref_out; int32_t* stop; double* rec;
    const double* w;   /* [B][8] ([B][7] Frenet) per-problem weights, or NULL: the handle's */
    /* mpcb200_solve_batch_frenet_on_path (frenet_on_path set; state and ref are NULL): the poses [B][4], the length of the path
     * ahead, e_y from the path or 0, and where K(s) and the solver's state go ([B][4] each, or NULL) */
    const double* pose; double window; int32_t ey_from_path;
    double* k_out; double* state_out;
    bool frenet_on_path;
};

/* doubles per weight row of a handle's model */
static size_t weight_row(int model) { return model ? 7 : 8; }

/* The per-problem arrays of a solve call, one table entry each.  The order is that of the packed small-batch layout
 * (solve_small_host): inputs, then warm (in and out), then outputs.  The last three belong to mpcb200_solve_batch_frenet_on_path
 * only, which never takes the packed path; the other calls never give them, so they leave the packed layout and the graph
 * key of those calls as they were. */
enum ArrayId { A_STATE, A_REF, A_PATH_OF, A_U_PREV, A_V_DES, A_W, A_WARM, A_U0, A_COST, A_TRAJ, A_STATUS, A_ITERS, A_REC, A_REF_OUT, A_STOP,
               A_POSE, A_K_OUT, A_STATE_OUT, A_COUNT };
enum { DIR_IN = 1, DIR_OUT = 2, DIR_INOUT = 3 };
/* an array's slot in the packed small-batch layout: there when the caller gives the array (PACK_GIVEN); always there and
 * copied, the kernel getting it only when given (PACK_SLOT); always there and always written by the kernel (PACK_ALWAYS), so
 * that one captured graph serves callers who ask for the output and callers who do not */
enum { PACK_GIVEN, PACK_SLOT, PACK_ALWAYS };
struct CallArray {
    char* host;     /* the caller's pointer, at the first problem of the slice (a device pointer for MPCB200_DEVICE); null: not given */
    size_t row;     /* bytes per problem */
    int dir;        /* DIR_* */
    int pack;       /* PACK_* */
    DevBuf* dev;    /* the handle's staging buffer for host pointers */
};

/* the table of a call's arrays from problem `lo` on, staged in handle h's buffers (d_ref also stages ref_out: on-path calls
 * have no ref) */
static void call_arrays(mpcb200_handle* h, const SolveArgs& a, int64_t lo, CallArray t[A_COUNT]) {
    const size_t d = sizeof(double), i4 = sizeof(int32_t);
    const size_t nt = (6 * (size_t)h->cfg.N + 4) * d, nr = 3 * ((size_t)h->cfg.N + 1) * d;
    const CallArray all[A_COUNT] = {
        {(char*)a.state, 4 * d, DIR_IN, PACK_GIVEN, &h->d_state},
        {(char*)a.ref, h->model ? 4 * d : nr, DIR_IN, PACK_GIVEN, &h->d_ref},
        {(char*)a.path_of, i4, DIR_IN, PACK_GIVEN, &h->d_pathof},
        {(char*)a.u_prev, 2 * d, DIR_IN, PACK_GIVEN, &h->d_uprev},
        {(char*)a.v_des, d, DIR_IN, PACK_SLOT, &h->d_vdes},
        {(char*)a.w, weight_row(h->model) * d, DIR_IN, PACK_GIVEN, &h->d_w},
        {(char*)a.warm, nt, DIR_INOUT, PACK_GIVEN, &h->d_warm},
        {(char*)a.u0, 2 * d, DIR_OUT, PACK_ALWAYS, &h->d_u0},
        {(char*)a.cost, d, DIR_OUT, PACK_ALWAYS, &h->d_cost},
        {(char*)a.traj, nt, DIR_OUT, PACK_SLOT, &h->d_traj},
        {(char*)a.status, i4, DIR_OUT, PACK_ALWAYS, &h->d_status},
        {(char*)a.iters, i4, DIR_OUT, PACK_ALWAYS, &h->d_iters},
        {(char*)a.rec, 4 * d, DIR_OUT, PACK_GIVEN, &h->d_rec},
        {(char*)a.ref_out, nr, DIR_OUT, PACK_GIVEN, &h->d_ref},
        {(char*)a.stop, i4, DIR_OUT, PACK_GIVEN, &h->d_stop},
        {(char*)a.pose, 4 * d, DIR_IN, PACK_GIVEN, &h->d_pose},
        {(char*)a.k_out, 4 * d, DIR_OUT, PACK_GIVEN, &h->d_ref},       /* (the call has no ref and no state) */
        {(char*)a.state_out, 4 * d, DIR_OUT, PACK_GIVEN, &h->d_state},
    };
    for (int i = 0; i < A_COUNT; i++) {
        t[i] = all[i];
        if (t[i].host) t[i].host += t[i].row * lo;
    }
}

/* the kernel arguments from one pointer per table entry (null: not in the call) */
static BatchPtrs batch_ptrs(void* const p[A_COUNT], int* resto, RefGen& rg) {
    rg.path_of = (const int*)p[A_PATH_OF]; rg.ref_out = (double*)p[A_REF_OUT]; rg.stop = (int*)p[A_STOP];
    return BatchPtrs{(const double*)p[A_STATE], (const double*)p[A_REF], (const double*)p[A_V_DES], (const double*)p[A_U_PREV],
                     (double*)p[A_WARM], (double*)p[A_U0], (double*)p[A_COST], (int*)p[A_STATUS], (int*)p[A_ITERS], (double*)p[A_TRAJ],
                     (double*)p[A_REC], resto, (const double*)p[A_W]};
}

/* The two least-squares fit matrices of the Frenet reference on this handle's device, [4][n1] then [4][n2] in d_fit, rebuilt and
 * uploaded when the window changes: grids of nav_msgs_path_frenet.py:63,79, arange(0, window, 0.5) and arange(0, window, 0.25) */
static int ensure_fit(mpcb200_handle* h, const char* who, double window) {
    if (h->fit_window == window) return MPCB200_OK;
    int n1, n2, rc;
    fit_grid_sizes(window, &n1, &n2);
    double* P = (double*)malloc(sizeof(double) * 4 * ((size_t)n1 + n2));
    if (!P) return fail(h, MPCB200_ENOMEM, "%s: out of host memory", who);
    cubic_fit_matrix(n1, 0.5, P); cubic_fit_matrix(n2, 0.25, P + 4 * (size_t)n1);
    rc = ensure(h, h->d_fit, sizeof(double) * 4 * ((size_t)n1 + n2));
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(h->d_fit.p, P, sizeof(double) * 4 * ((size_t)n1 + n2), cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) rc = fail(h, MPCB200_ECUDA, "%s: %s", who, cudaGetErrorString(e));
    }
    free(P);
    if (rc) return rc;
    h->fit_window = window; h->fit_n1 = n1; h->fit_n2 = n2;
    return MPCB200_OK;
}

/* mpcb200_solve_batch_frenet_on_path on one device: on_path_frenet_ref_kernel, launch_solve on the rows it wrote (an ordinary
 * Frenet batch: the kernel and layout mpcb200_solve_batch_frenet would take), then on_path_invalid_kernel for the problems whose
 * path id was never set.  p: the call's arrays on this device, io / rg as batch_ptrs made them from p (rg: this device's tables) */
static int launch_frenet_on_path(mpcb200_handle* h, int64_t B, const SolveArgs& a, void* const p[A_COUNT], BatchPtrs io, const RefGen& rg) {
    int rc;
    if ((rc = ensure_fit(h, a.who, a.window))) return rc;
    const size_t rows = (size_t)B * 4 * sizeof(double);
    double* k_out = (double*)p[A_K_OUT];
    double* state_out = (double*)p[A_STATE_OUT];
    double* vdes = nullptr;
    if (!k_out) { if ((rc = ensure(h, h->d_ref, rows))) return rc; k_out = (double*)h->d_ref.p; }
    if (!state_out) { if ((rc = ensure(h, h->d_state, rows))) return rc; state_out = (double*)h->d_state.p; }
    if (!io.v_des) { if ((rc = ensure(h, h->d_vdes, (size_t)B * sizeof(double)))) return rc; vdes = (double*)h->d_vdes.p; }
    FrenetRolloutArgs fa;
    memset(&fa, 0, sizeof(fa));
    for (int i = 0; i < 3; i++) fa.paths[i] = rg.paths[i];
    fa.path_of = rg.path_of; fa.B = (long)B; fa.ey_from_path = a.ey_from_path;
    fa.P1 = (const double*)h->d_fit.p; fa.P2 = fa.P1 + 4 * (size_t)h->fit_n1; fa.n1 = h->fit_n1; fa.n2 = h->fit_n2;
    const long long wblocks = (B + 3) / 4, wmax = (long long)h->num_sms * 16;
    on_path_frenet_ref_kernel<<<(int)(wblocks < wmax ? wblocks : wmax), 128, 0, h->stream>>>(make_kcfg(h), fa, (const double*)p[A_POSE],
                                                                                             k_out, state_out, vdes, a.target_vel);
    CUDA_TRY(h, cudaGetLastError());
    h->stats.kernel_launches += 1;
    io.state = state_out; io.ref = k_out;
    if (vdes) io.v_des = vdes;
    RefGen none;
    memset(&none, 0, sizeof(none));
    if ((rc = launch_solve(h, B, io, none))) return rc;
    on_path_invalid_kernel<<<(int)((B + 127) / 128), 128, 0, h->stream>>>((long long)B, rg, io);
    CUDA_TRY(h, cudaGetLastError());
    h->stats.kernel_launches += 1;
    return MPCB200_OK;
}

/* contiguous slice of `total` owned by part `i` of `parts`; sizes differ by at most one (same rule as sharding.shard_range) */
static void shard_range(int64_t total, int parts, int i, int64_t* lo, int64_t* hi) {
    const int64_t base = total / parts, rem = total % parts;
    *lo = i * base + (i < rem ? i : rem);
    *hi = *lo + base + (i < rem ? 1 : 0);
}

/* Host pointers on a multi-GPU handle: one contiguous slice [lo[i], hi[i]) of the B problems per device dev[i] of the first
 * n_dev, all working at once (one slice when there are fewer than two problems per device).  Clears the stats of the sub-handles
 * that get a slice; returns the number of slices. */
static int slice_call(mpcb200_handle* h, int64_t B, int n_dev, mpcb200_handle* dev[8], int64_t lo[8], int64_t hi[8]) {
    const int parts = (B >= 2 * (int64_t)n_dev) ? n_dev : 1;
    dev[0] = h;
    for (int i = 0; i < h->n_sub; i++) dev[i + 1] = h->sub[i];
    for (int i = 0; i < parts; i++) {
        shard_range(B, parts, i, &lo[i], &hi[i]);
        if (i) memset(&dev[i]->stats, 0, sizeof(mpcb200_stats));
    }
    return parts;
}

/* the sub-handles' counters into the handle the caller holds */
static void merge_stats(mpcb200_handle* h, mpcb200_handle* const dev[8], int parts) {
    for (int i = 1; i < parts; i++) {
        h->stats.kernel_launches += dev[i]->stats.kernel_launches;
        h->stats.h2d_bytes += dev[i]->stats.h2d_bytes; h->stats.d2h_bytes += dev[i]->stats.d2h_bytes;
        if (dev[i]->stats.kernel_ms > h->stats.kernel_ms) h->stats.kernel_ms = dev[i]->stats.kernel_ms;   /* the devices run concurrently */
    }
}

/* host path ids: each one set with mpcb200_set_path (`what`: "problem" or "vehicle") */
static int check_path_ids(mpcb200_handle* h, const char* who, const char* what, int64_t B, const int32_t* path_of) {
    for (int64_t b = 0; b < B; b++)
        if (path_of[b] < 0 || path_of[b] > 2 || h->path_n[path_of[b]] == 0)
            return fail(h, MPCB200_EINVAL, "%s: %s %lld uses path %d, which was not set with mpcb200_set_path", who, what, (long long)b, path_of[b]);
    return MPCB200_OK;
}

/* host weight rows of nw doubles: mpcb200_set_cost's rule (device rows are checked by the kernel: MPCB200_ERROR for that problem) */
static int check_weight_rows(mpcb200_handle* h, const char* who, const char* what, int64_t B, const double* w, size_t nw) {
    for (int64_t b = 0; b < B; b++)
        for (size_t i = 0; i < nw; i++)
            if (!(w[b * nw + i] >= 0.0)) return fail(h, MPCB200_EINVAL, "%s: weight %d of %s %lld is negative or NaN", who, (int)i, what, (long long)b);
    return MPCB200_OK;
}

/* Host pointers, small batch (the control loop's batch of one): latency is the driver calls, not the bytes.  All
 * inputs are packed into one pinned buffer (with the zeroed problem counter in front) and go over in ONE copy, all
 * outputs come back in ONE copy: 7 driver calls instead of ~16. */
static const int64_t SMALL_BATCH = 64;
static int solve_small_host(mpcb200_handle* h, int64_t B, const SolveArgs& a) {
    CallArray t[A_COUNT];
    call_arrays(h, a, 0, t);
    /* layout in doubles: [counter, pad] inputs | warm | outputs, each slot a whole number of doubles, the restoration counts
     * just before rec.  in_end: the end of what is copied in, out_from: the start of what is copied out (the warm slot is in both) */
    size_t off[A_COUNT], o = 2, in_end = 2, out_from = 0, o_resto = 0;
    for (int i = 0; i < A_COUNT; i++) {
        if (i == A_REC) { o_resto = o; o += (B + 1) / 2; }
        off[i] = o;
        if (!t[i].host && t[i].pack == PACK_GIVEN) continue;
        if ((t[i].dir & DIR_OUT) && !out_from) out_from = o;
        o += (t[i].row * B + sizeof(double) - 1) / sizeof(double);
        if (t[i].dir & DIR_IN) in_end = o;
    }
    const size_t total = o, bytes = total * sizeof(double);
    int rc;
    if (bytes > h->d_stage.cap || bytes > h->h_stage_cap) drop_graphs(h);   /* the graphs hold the old addresses */
    if ((rc = ensure(h, h->d_stage, bytes))) return rc;
    if (bytes > h->h_stage_cap) {
        if (h->h_stage) CUDA_TRY(h, cudaFreeHost(h->h_stage));
        h->h_stage = nullptr; h->h_stage_cap = 0;
        CUDA_TRY(h, cudaHostAlloc(&h->h_stage, bytes + bytes / 4, cudaHostAllocDefault));
        h->h_stage_cap = bytes + bytes / 4;
    }
    double* hs = (double*)h->h_stage;
    double* ds = (double*)h->d_stage.p;
    hs[0] = 0.0; hs[1] = 0.0;   /* the problem counter (all-zero bits) */
    void* p[A_COUNT];
    int flags = 0;   /* the graph's shape: which arrays the kernel gets (the rows of w are data) */
    for (int i = 0; i < A_COUNT; i++) {
        if (t[i].host && (t[i].dir & DIR_IN)) memcpy(hs + off[i], t[i].host, t[i].row * B);
        p[i] = (t[i].host || t[i].pack == PACK_ALWAYS) ? ds + off[i] : nullptr;
        if (t[i].host && t[i].pack != PACK_ALWAYS) flags |= 1 << i;
    }
    cudaStream_t s = h->stream;
    RefGen rg;
    memset(&rg, 0, sizeof(rg));
    const BatchPtrs io = batch_ptrs(p, (int*)(ds + o_resto), rg);
    /* the sequence copy in -> kernel -> copy out; `ext`: events recorded from inside a graph need the external flag to be timed */
    auto enqueue = [&](bool ext) -> int {
        CUDA_TRY(h, cudaMemcpyAsync(ds, hs, in_end * sizeof(double), cudaMemcpyHostToDevice, s));
        CUDA_TRY(h, cudaEventRecordWithFlags(h->ev0, s, ext ? cudaEventRecordExternal : cudaEventRecordDefault));
        int r = launch_solve(h, B, io, rg, (unsigned long long*)ds);
        if (r) return r;
        CUDA_TRY(h, cudaEventRecordWithFlags(h->ev1, s, ext ? cudaEventRecordExternal : cudaEventRecordDefault));
        CUDA_TRY(h, cudaMemcpyAsync(hs + out_from, ds + out_from, (total - out_from) * sizeof(double), cudaMemcpyDeviceToHost, s));
        return 0;
    };
    bool launched = false;
    if (h->graphs_ok && s == h->own_stream) {
        cudaGraphExec_t exec = nullptr;
        for (int i = 0; i < h->n_graphs; i++) if (h->graphs[i].B == B && h->graphs[i].flags == flags) exec = h->graphs[i].exec;
        if (!exec) {
            cudaGraph_t graph = nullptr;
            bool ok = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            if (ok) {
                const int r = enqueue(true);
                ok = (cudaStreamEndCapture(s, &graph) == cudaSuccess) && r == 0 && graph != nullptr;
                h->stats.kernel_launches = 0;   /* counted at the graph launch below */
            }
            if (ok) ok = cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
            if (graph) cudaGraphDestroy(graph);
            if (ok) {
                if (h->n_graphs == 8) drop_graphs(h);
                h->graphs[h->n_graphs].B = B; h->graphs[h->n_graphs].flags = flags; h->graphs[h->n_graphs].exec = exec;
                h->n_graphs++;
            } else {
                exec = nullptr; h->graphs_ok = false; cudaGetLastError();   /* fall back to plain launches for good */
            }
        }
        if (exec) {
            if (cudaGraphLaunch(exec, s) == cudaSuccess) { launched = true; h->stats.kernel_launches += 1; }
            else { h->graphs_ok = false; cudaGetLastError(); drop_graphs(h); }
        }
    }
    if (!launched && (rc = enqueue(false))) return rc;
    h->stats.h2d_bytes += in_end * sizeof(double);
    h->stats.d2h_bytes += (total - out_from) * sizeof(double);
    CUDA_TRY(h, cudaStreamSynchronize(s));
    for (int i = 0; i < A_COUNT; i++)
        if (t[i].host && (t[i].dir & DIR_OUT)) memcpy(t[i].host, hs + off[i], t[i].row * B);
    memcpy(h->small_resto, hs + o_resto, B * sizeof(int32_t));   /* where mpcb200_get_restorations looks after a small batch */
    h->resto_on_host = true;
    float ms = 0.f;
    CUDA_TRY(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->stats.kernel_ms = ms;
    return MPCB200_OK;
}

/* HOST pointers, one device: stage the slice through the handle's device buffers and launch (asynchronous) ... */
static int host_enqueue(mpcb200_handle* h, int64_t B, const SolveArgs& a, int64_t lo, const RefGen& rg0) {
    CUDA_TRY(h, cudaSetDevice(h->device));
    CallArray t[A_COUNT];
    call_arrays(h, a, lo, t);
    int rc;
    for (int i = 0; i < A_COUNT; i++)
        if (t[i].host && (rc = ensure(h, *t[i].dev, t[i].row * B))) return rc;
    if ((rc = ensure(h, h->d_resto, B * sizeof(int32_t)))) return rc;
    cudaStream_t s = h->stream;
    void* p[A_COUNT];
    for (int i = 0; i < A_COUNT; i++) {
        p[i] = t[i].host ? t[i].dev->p : nullptr;
        if (!t[i].host || !(t[i].dir & DIR_IN)) continue;
        CUDA_TRY(h, cudaMemcpyAsync(p[i], t[i].host, t[i].row * B, cudaMemcpyHostToDevice, s));
        h->stats.h2d_bytes += t[i].row * B;
    }
    RefGen rg = rg0;
    if (a.path_of) fill_paths(h, rg.paths);   /* this device's copies of the tables */
    const BatchPtrs io = batch_ptrs(p, (int*)h->d_resto.p, rg);
    CUDA_TRY(h, cudaEventRecord(h->ev0, s));
    if ((rc = a.frenet_on_path ? launch_frenet_on_path(h, B, a, p, io, rg) : launch_solve(h, B, io, rg))) return rc;
    CUDA_TRY(h, cudaEventRecord(h->ev1, s));
    return MPCB200_OK;
}

/* ... and bring the slice's results back into the caller's buffers (synchronises the device's stream) */
static int host_collect(mpcb200_handle* h, int64_t B, const SolveArgs& a, int64_t lo) {
    CUDA_TRY(h, cudaSetDevice(h->device));
    CallArray t[A_COUNT];
    call_arrays(h, a, lo, t);
    cudaStream_t s = h->stream;
    for (int i = 0; i < A_COUNT; i++) {
        if (!t[i].host || !(t[i].dir & DIR_OUT)) continue;
        CUDA_TRY(h, cudaMemcpyAsync(t[i].host, t[i].dev->p, t[i].row * B, cudaMemcpyDeviceToHost, s));
        h->stats.d2h_bytes += t[i].row * B;
    }
    CUDA_TRY(h, cudaStreamSynchronize(s));
    float ms = 0.f;
    CUDA_TRY(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->stats.kernel_ms = ms;
    return MPCB200_OK;
}

/* a sub-handle's error text and counters surface through the handle the caller holds */
static int sub_fail(mpcb200_handle* h, mpcb200_handle* d, int rc) {
    if (d != h) snprintf(h->err, sizeof(h->err), "device %d: %.400s", d->device, d->err);
    return rc;
}

/* common body of mpcb200_solve_batch* (ref given), mpcb200_solve_batch_on_path (path_of given) and mpcb200_solve_batch_frenet_on_path
 * (pose and path_of given) */
static int solve_batch_impl(mpcb200_handle* h, int64_t B, const SolveArgs& a, int32_t mem_space) {
    const char* who = a.who;
    if (!h) return MPCB200_EINVAL;
    if (B < 0) return fail(h, MPCB200_EINVAL, "%s: B=%lld", who, (long long)B);
    if (mem_space != MPCB200_HOST && mem_space != MPCB200_DEVICE) return fail(h, MPCB200_EINVAL, "%s: mem_space=%d", who, mem_space);
    memset(&h->stats, 0, sizeof(h->stats));
    h->last_B = B; h->last_sharded = false; h->resto_on_host = false;
    if (B == 0) return MPCB200_OK;
    const bool on_path = (a.path_of != nullptr);
    if (a.frenet_on_path) {
        if (!a.pose || !a.path_of || !a.u_prev || !a.u0) return fail(h, MPCB200_EINVAL, "%s: pose, path_of, u_prev and u0 are required", who);
    } else if (!a.state || (!a.ref && !on_path) || !a.u_prev || (!a.u0 && !a.rec))
        return fail(h, MPCB200_EINVAL, "%s: state, %s, u_prev and %s are required", who, on_path ? "path_of" : "ref", a.rec ? "rec" : "u0");
    if (on_path && h->model && !a.frenet_on_path) return fail(h, MPCB200_EINVAL, "%s: not available for the Frenet-frame variant", who);
    int rc;
    if (a.w && mem_space == MPCB200_HOST && (rc = check_weight_rows(h, who, "problem", B, a.w, weight_row(h->model)))) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    RefGen rg;
    memset(&rg, 0, sizeof(rg));
    if (on_path) {
        fill_paths(h, rg.paths);
        rg.track_using_time = a.track_using_time;
        rg.target_vel = a.target_vel > 0.0 ? a.target_vel : 0.0;   /* des_speed, mpc_cmd_pub.jl:58-62 */
        if (mem_space == MPCB200_HOST && (rc = check_path_ids(h, who, "problem", B, a.path_of))) return rc;
    }
    if (mem_space == MPCB200_DEVICE) {
        if ((rc = ensure(h, h->d_resto, B * sizeof(int32_t)))) return rc;
        CallArray t[A_COUNT];
        call_arrays(h, a, 0, t);
        void* p[A_COUNT];
        for (int i = 0; i < A_COUNT; i++) p[i] = t[i].host;
        const BatchPtrs io = batch_ptrs(p, (int*)h->d_resto.p, rg);
        return a.frenet_on_path ? launch_frenet_on_path(h, B, a, p, io, rg) : launch_solve(h, B, io, rg);
    }
    if (!on_path && B <= SMALL_BATCH) return solve_small_host(h, B, a);
    mpcb200_handle* dev[8];
    const int parts = slice_call(h, B, h->n_sub + 1, dev, h->slice_lo, h->slice_hi);
    for (int i = 0; i < parts; i++)
        if ((rc = host_enqueue(dev[i], h->slice_hi[i] - h->slice_lo[i], a, h->slice_lo[i], rg))) return sub_fail(h, dev[i], rc);
    for (int i = 0; i < parts; i++)
        if ((rc = host_collect(dev[i], h->slice_hi[i] - h->slice_lo[i], a, h->slice_lo[i]))) return sub_fail(h, dev[i], rc);
    merge_stats(h, dev, parts);
    h->last_sharded = parts > 1;
    for (int i = parts; i < 8; i++) h->slice_lo[i] = h->slice_hi[i] = 0;
    CUDA_TRY(h, cudaSetDevice(h->device));
    return MPCB200_OK;
}

int mpcb200_get_restorations(mpcb200_handle* h, int64_t B, int32_t* out) {
    if (!h || !out) return fail(h, MPCB200_EINVAL, "mpcb200_get_restorations: NULL argument");
    if (B != h->last_B) return fail(h, MPCB200_EINVAL, "mpcb200_get_restorations: B=%lld, the last solve had %lld problems", (long long)B, (long long)h->last_B);
    if (B == 0) return MPCB200_OK;
    if (h->resto_on_host) { memcpy(out, h->small_resto, B * sizeof(int32_t)); return MPCB200_OK; }
    if (!h->last_sharded) {
        CUDA_TRY(h, cudaSetDevice(h->device));
        CUDA_TRY(h, cudaMemcpyAsync(out, h->d_resto.p, B * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        return MPCB200_OK;
    }
    for (int i = 0; i <= h->n_sub; i++) {
        mpcb200_handle* d = i ? h->sub[i - 1] : h;
        const int64_t n = h->slice_hi[i] - h->slice_lo[i];
        if (n <= 0) continue;
        CUDA_TRY(h, cudaSetDevice(d->device));
        CUDA_TRY(h, cudaMemcpyAsync(out + h->slice_lo[i], d->d_resto.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, d->stream));
        CUDA_TRY(h, cudaStreamSynchronize(d->stream));
    }
    CUDA_TRY(h, cudaSetDevice(h->device));
    return MPCB200_OK;
}

/* mpcb200_solve_batch_frenet and mpcb200_solve_batch_frenet_w (w == NULL: the handle's weights) */
static int solve_frenet(const char* who, mpcb200_handle* h, int64_t B, const double* state, const double* k_coeffs, const double* v_des,
                        const double* u_prev, double* warm, const double* w, double* u0, double* cost, int32_t* status, int32_t* iters,
                        double* traj, int32_t mem_space) {
    if (h && !h->model) return fail(h, MPCB200_EINVAL, "%s: the handle was not created with mpcb200_create_frenet", who);
    const SolveArgs a{who, state, k_coeffs, nullptr, 1, 0.0, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, nullptr, nullptr, w};
    return solve_batch_impl(h, B, a, mem_space);
}

int mpcb200_solve_batch_frenet(mpcb200_handle* h, int64_t B, const double* state, const double* k_coeffs, const double* v_des,
                               const double* u_prev, double* warm, double* u0, double* cost, int32_t* status, int32_t* iters,
                               double* traj, int32_t mem_space) {
    return solve_frenet("mpcb200_solve_batch_frenet", h, B, state, k_coeffs, v_des, u_prev, warm, nullptr, u0, cost, status, iters, traj, mem_space);
}

int mpcb200_solve_batch_frenet_w(mpcb200_handle* h, int64_t B, const double* state, const double* k_coeffs, const double* v_des,
                                 const double* u_prev, double* warm, const double* w, double* u0, double* cost, int32_t* status,
                                 int32_t* iters, double* traj, int32_t mem_space) {
    if (h && !w) return fail(h, MPCB200_EINVAL, "mpcb200_solve_batch_frenet_w: w is required");
    return solve_frenet("mpcb200_solve_batch_frenet_w", h, B, state, k_coeffs, v_des, u_prev, warm, w, u0, cost, status, iters, traj, mem_space);
}

int mpcb200_set_cost_frenet(mpcb200_handle* h, const double w[7]) {
    if (!h || !w) return fail(h, MPCB200_EINVAL, "mpcb200_set_cost_frenet: NULL argument");
    if (!h->model) return fail(h, MPCB200_EINVAL, "mpcb200_set_cost_frenet: the handle was not created with mpcb200_create_frenet");
    for (int i = 0; i < 7; i++) if (!(w[i] >= 0.0)) return fail(h, MPCB200_EINVAL, "mpcb200_set_cost_frenet: weight %d is negative or NaN", i);
    h->w[0] = 0.0;
    memcpy(h->w + 1, w, 7 * sizeof(double));
    drop_graphs(h);
    for (int i = 0; i < h->n_sub; i++) { memcpy(h->sub[i]->w, h->w, 8 * sizeof(double)); drop_graphs(h->sub[i]); }
    return MPCB200_OK;
}

/* mpcb200_solve_batch and mpcb200_solve_batch_w (w == NULL: the handle's weights) */
static int solve_xy(const char* who, mpcb200_handle* h, int64_t B, const double* state, const double* ref, const double* v_des,
                    const double* u_prev, double* warm, const double* w, double* u0, double* cost, int32_t* status, int32_t* iters,
                    double* traj, int32_t mem_space) {
    if (h && h->model) return fail(h, MPCB200_EINVAL, "%s: Frenet handle; use mpcb200_solve_batch_frenet", who);
    const SolveArgs a{who, state, ref, nullptr, 1, 0.0, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, nullptr, nullptr, w};
    return solve_batch_impl(h, B, a, mem_space);
}

int mpcb200_solve_batch(mpcb200_handle* h, int64_t B, const double* state, const double* ref, const double* v_des,
                        const double* u_prev, double* warm, double* u0, double* cost, int32_t* status, int32_t* iters,
                        double* traj, int32_t mem_space) {
    return solve_xy("mpcb200_solve_batch", h, B, state, ref, v_des, u_prev, warm, nullptr, u0, cost, status, iters, traj, mem_space);
}

int mpcb200_solve_batch_w(mpcb200_handle* h, int64_t B, const double* state, const double* ref, const double* v_des,
                          const double* u_prev, double* warm, const double* w, double* u0, double* cost, int32_t* status,
                          int32_t* iters, double* traj, int32_t mem_space) {
    if (h && !w) return fail(h, MPCB200_EINVAL, "mpcb200_solve_batch_w: w is required");
    return solve_xy("mpcb200_solve_batch_w", h, B, state, ref, v_des, u_prev, warm, w, u0, cost, status, iters, traj, mem_space);
}

int mpcb200_solve_batch_records(mpcb200_handle* h, int64_t B, const double* state, const double* ref, const double* v_des,
                                const double* u_prev, double* warm, double* rec, double* traj, int32_t mem_space) {
    if (h && !rec) return fail(h, MPCB200_EINVAL, "mpcb200_solve_batch_records: rec is required");
    /* u0 is part of the record; the kernel still wants a place for it in DEVICE mode: none is needed, it skips NULL */
    const SolveArgs a{"mpcb200_solve_batch_records", state, ref, nullptr, 1, 0.0, v_des, u_prev, warm, nullptr, nullptr, nullptr, nullptr, traj,
                      nullptr, nullptr, rec};
    return solve_batch_impl(h, B, a, mem_space);
}

int mpcb200_solve_batch_on_path(mpcb200_handle* h, int64_t B, const double* state, const int32_t* path_of, int32_t track_using_time,
                                double target_vel, const double* v_des, const double* u_prev, double* warm, double* u0, double* cost,
                                int32_t* status, int32_t* iters, double* traj, double* ref_out, int32_t* stop, int32_t mem_space) {
    if (h && !path_of) return fail(h, MPCB200_EINVAL, "mpcb200_solve_batch_on_path: path_of is required");
    const SolveArgs a{"mpcb200_solve_batch_on_path", state, nullptr, path_of, track_using_time, target_vel, v_des, u_prev, warm, u0, cost,
                      status, iters, traj, ref_out, stop, nullptr};
    return solve_batch_impl(h, B, a, mem_space);
}

int mpcb200_solve_batch_frenet_on_path(mpcb200_handle* h, int64_t B, const double* pose, const int32_t* path_of, double window,
                                       double target_vel, int32_t ey_from_path, const double* v_des, const double* u_prev, double* warm,
                                       const double* w, double* u0, double* cost, int32_t* status, int32_t* iters, double* traj,
                                       double* k_coeffs_out, double* state_out, int32_t mem_space) {
    const char* who = "mpcb200_solve_batch_frenet_on_path";
    if (h && !h->model) return fail(h, MPCB200_EINVAL, "%s: the handle was not created with mpcb200_create_frenet", who);
    if (h && !(window >= 4.0 && window <= 500.0)) return fail(h, MPCB200_EINVAL, "%s: window %.3g m outside [4, 500]", who, window);
    const SolveArgs a{who, nullptr, nullptr, path_of, 0, target_vel, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, nullptr,
                      nullptr, w, pose, window, ey_from_path, k_coeffs_out, state_out, true};
    return solve_batch_impl(h, B, a, mem_space);
}

int mpcb200_set_path(mpcb200_handle* h, int32_t path_id, int32_t n, const double* t, const double* X, const double* Y,
                     const double* psi, const double* s) {
    if (!h) return MPCB200_EINVAL;
    if (path_id < 0 || path_id > 2) return fail(h, MPCB200_EINVAL, "mpcb200_set_path: path_id %d outside [0,2]", path_id);
    if (n < 2 || !t || !X || !Y || !psi || !s) return fail(h, MPCB200_EINVAL, "mpcb200_set_path: need n >= 2 samples and five columns");
    CUDA_TRY(h, cudaSetDevice(h->device));
    const int nch = path_chunks(n);
    int rc = ensure(h, h->d_path[path_id], ((size_t)5 * n + (size_t)3 * nch) * sizeof(double));
    if (rc) return rc;
    const double* cols[5] = {t, X, Y, psi, s};
    for (int i = 0; i < 5; i++)
        CUDA_TRY(h, cudaMemcpyAsync((double*)h->d_path[path_id].p + (size_t)i * n, cols[i], (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    /* bounding circles of the chunks of samples the nearest-sample search skips (TeamSolver::nearest_sample) */
    double* cb = (double*)malloc((size_t)3 * nch * sizeof(double));
    if (!cb) return fail(h, MPCB200_ENOMEM, "mpcb200_set_path: out of host memory");
    path_chunk_bounds(n, X, Y, cb);
    const cudaError_t ce = cudaMemcpyAsync((double*)h->d_path[path_id].p + (size_t)5 * n, cb, (size_t)3 * nch * sizeof(double), cudaMemcpyHostToDevice, h->stream);
    const cudaError_t cs = cudaStreamSynchronize(h->stream);
    free(cb);
    CUDA_TRY(h, ce);
    CUDA_TRY(h, cs);
    h->path_n[path_id] = n;
    for (int i = 0; i < h->n_sub; i++)   /* the tables are replicated on every device */
        if ((rc = mpcb200_set_path(h->sub[i], path_id, n, t, X, Y, psi, s))) return sub_fail(h, h->sub[i], rc);
    if (h->n_sub) CUDA_TRY(h, cudaSetDevice(h->device));
    return MPCB200_OK;
}

/* The start point of a vehicle's FIRST solve: the solution of the module-load solve of the default problem
 * (MKZMPCPathFollower.jl:36-39,75,82,110-113,126-128: zero state and previous command, x_ref = 15 t, y_ref = psi_ref = 0,
 * module-default weights, start = 0.0), which JuMP re-solves from.  Solved once per handle with this library. */
static int ensure_seed(mpcb200_handle* h) {
    if (h->seed_valid) return MPCB200_OK;
    const int N = h->cfg.N;
    const size_t nt = 6 * (size_t)N + 4;
    double* buf = (double*)calloc(4 + 3 * ((size_t)N + 1) + 2 + 1 + 2 + nt, sizeof(double));
    if (!buf) return fail(h, MPCB200_ENOMEM, "mpcb200_rollout: out of host memory");
    double *state = buf, *ref = state + 4, *u_prev = ref + 3 * (N + 1), *v_des = u_prev + 2, *u0 = v_des + 1, *traj = u0 + 2;
    for (int k = 0; k <= N; k++) ref[k] = 15.0 * ((double)k * h->cfg.dt);
    v_des[0] = 15.0;
    double w_keep[8];
    memcpy(w_keep, h->w, sizeof(w_keep));
    memcpy(h->w, W_XY_DEFAULT, sizeof(W_XY_DEFAULT));
    const int start_keep = h->cfg.start_mode;
    h->cfg.start_mode = MPCB200_START_ZERO;
    drop_graphs(h);   /* weights and start mode are kernel parameters */
    const mpcb200_stats keep = h->stats;
    const SolveArgs a{"mpcb200_rollout (module-load solve)", state, ref, nullptr, 1, 0.0, v_des, u_prev, nullptr, u0, nullptr, nullptr, nullptr,
                      traj, nullptr, nullptr, nullptr};
    int rc = solve_small_host(h, 1, a);
    memcpy(h->w, w_keep, sizeof(w_keep));
    h->cfg.start_mode = start_keep;
    drop_graphs(h);
    h->stats = keep;
    if (!rc) rc = ensure(h, h->d_seed, nt * sizeof(double));
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(h->d_seed.p, traj, nt * sizeof(double), cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) rc = fail(h, MPCB200_ECUDA, "mpcb200_rollout: %s", cudaGetErrorString(e));
    }
    free(buf);
    if (!rc) h->seed_valid = true;
    return rc;
}

/* one closed-loop call: mpcb200_rollout and mpcb200_rollout_w (model 0) or mpcb200_rollout_frenet and mpcb200_rollout_frenet_w (model 1) */
struct RolloutCall {
    const char* who;
    int model;
    int64_t B; int32_t T;
    const double* pose0; const int32_t* path_of;
    double target_vel;
    int32_t track_using_time; const double* w;   /* XY: waypoints by time or arc length; [B][8] ([B][7] Frenet) weight rows or null */
    double window; int32_t ey_from_path;          /* Frenet: length of the path ahead, e_y from the path or from the fit */
    double* log; double* final_state;             /* [T][B][8], [B][8] or null */
    double* metrics;                              /* [B][MET_FIELDS] or null (the plain entry points) */
};

/* one device's share of a rollout: vehicles [lo, lo + n) of B; enqueue ... */
static int rollout_enqueue(mpcb200_handle* h, const RolloutCall& c, int64_t lo, int64_t n) {
    CUDA_TRY(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    int rc;
    if (!c.model && (rc = ensure_seed(h))) return rc;
    if (c.model && (rc = ensure_fit(h, c.who, c.window))) return rc;
    if ((rc = ensure(h, h->d_pose, (size_t)n * 3 * sizeof(double)))) return rc;
    if ((rc = ensure(h, h->d_pathof, (size_t)n * sizeof(int32_t)))) return rc;
    if (c.log && (rc = ensure(h, h->d_log, (size_t)c.T * n * 8 * sizeof(double)))) return rc;
    if (c.final_state && (rc = ensure(h, h->d_final, (size_t)n * 8 * sizeof(double)))) return rc;
    const long long Bp = (n + 31) / 32 * 32;   /* stride of the per-period pipeline's structure-of-arrays buffers */
    if (c.metrics && ((rc = ensure(h, h->d_met, (size_t)MET_K * Bp * sizeof(double))) ||
                      (rc = ensure(h, h->d_metout, (size_t)n * MET_FIELDS * sizeof(double))))) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(h->d_pose.p, c.pose0 + 3 * lo, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice, s));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_pathof.p, c.path_of + lo, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    h->stats.h2d_bytes += (size_t)n * (3 * sizeof(double) + sizeof(int32_t));
    if (c.w) {
        const size_t nw = c.model ? 7 : 8;
        if ((rc = ensure(h, h->d_w, (size_t)n * nw * sizeof(double)))) return rc;
        CUDA_TRY(h, cudaMemcpyAsync(h->d_w.p, c.w + nw * lo, (size_t)n * nw * sizeof(double), cudaMemcpyHostToDevice, s));
        h->stats.h2d_bytes += (size_t)n * nw * sizeof(double);
    }
    /* the kernel arguments of both models; only those of c.model are launched with */
    RolloutArgs a;
    FrenetRolloutArgs fa;
    memset(&a, 0, sizeof(a));
    memset(&fa, 0, sizeof(fa));
    a.pose0 = fa.pose0 = (const double*)h->d_pose.p; a.path_of = fa.path_of = (const int*)h->d_pathof.p;
    fill_paths(h, a.paths); fill_paths(h, fa.paths);
    a.T = fa.T = c.T; a.target_vel = fa.target_vel = c.target_vel; a.B = fa.B = (long)n;
    a.log = fa.log = c.log ? (double*)h->d_log.p : nullptr; a.final_state = fa.final_state = c.final_state ? (double*)h->d_final.p : nullptr;
    a.track_using_time = c.track_using_time; a.warm0 = (const double*)h->d_seed.p; a.w = c.w ? (const double*)h->d_w.p : nullptr;
    fa.ey_from_path = c.ey_from_path;
    fa.P1 = (const double*)h->d_fit.p; fa.P2 = fa.P1 + 4 * (size_t)h->fit_n1; fa.n1 = h->fit_n1; fa.n2 = h->fit_n2;
    a.met = c.metrics ? (double*)h->d_met.p : nullptr;
    const KCfg kc = make_kcfg(h);
    /* large fleets at short horizons: one control period = plant / reference / thread-per-problem solve over the whole fleet.
     * Measured for the XY model at N = 8, 200 periods (profiles/r02_logs/r02_rollout_thresholds.log): a period of the pipeline takes
     * ~0.9 ms up to 8,192 vehicles (the slowest vehicle's dozen solver trips) and grows slowly after that, the fused kernel takes
     * 0.5 / 0.8 / 1.4 / 2.5 ms at 2,048 / 4,096 / 8,192 / 16,384 vehicles: the default rule switches at a quarter of the cold-start batch */
    const int64_t roll_from = h->tpp_default_rule ? h->tpp_min_batch / 4 : h->tpp_min_batch;
    if (h->tpp_min_batch > 0 && n >= roll_from) {
        /* blocks of 128 vehicles (two resident per SM): every vehicle solves at once and a block keeps its vehicles, so smaller
         * blocks mean less idle SMs in the last wave (16,384 vehicles: 0.89 instead of 1.07 ms per period; never slower) */
        const int tb = h->tpp_block < 128 ? h->tpp_block : 128;
        const long long sblocks = (n + tb - 1) / tb, S = sblocks * tb;
        /* vehicle state [RV_NF][Bp], then for the Frenet model the reference of the period [6][Bp] */
        const size_t veh_rows = c.model ? RV_NF + 6 : RV_NF;
        if ((rc = ensure(h, h->d_tpp_state, tpp_state_doubles(h->cfg.N, (long)S, c.model) * sizeof(double)))) return rc;
        if ((rc = ensure(h, h->d_tpp_filt, tpp_filter_doubles((long)S) * sizeof(double)))) return rc;
        if ((rc = ensure(h, h->d_veh, veh_rows * Bp * sizeof(double)))) return rc;
        if (!c.model && (rc = ensure(h, h->d_vstop, (size_t)Bp * sizeof(int)))) return rc;
        if ((rc = ensure(h, h->d_u0, (size_t)n * 2 * sizeof(double)))) return rc;
        if ((rc = ensure(h, h->d_status, (size_t)n * sizeof(int32_t)))) return rc;
        if ((rc = ensure(h, h->d_iters, (size_t)n * sizeof(int32_t)))) return rc;
        BatchPtrs out;
        memset(&out, 0, sizeof(out));
        out.u0 = (double*)h->d_u0.p; out.status = (int*)h->d_status.p; out.iters = (int*)h->d_iters.p; out.w = a.w;
        auto sk = c.model ? (a.w ? rollout_solve_tpp_kernel<1, 1> : rollout_solve_tpp_kernel<1, 0>)
                          : (a.w ? rollout_solve_tpp_kernel<0, 1> : rollout_solve_tpp_kernel<0, 0>);
        RefGen rg;
        memset(&rg, 0, sizeof(rg));
        fill_paths(h, rg.paths);
        rg.track_using_time = c.track_using_time;
        /* XY: des_speed of mpc_cmd_pub.jl:58-62; the Frenet node uses its target speed as given */
        const double des_speed = (c.model || c.target_vel > 0.0) ? c.target_vel : 0.0;
        rg.target_vel = des_speed;
        double* veh = (double*)h->d_veh.p;
        double* fref = c.model ? veh + (size_t)RV_NF * Bp : nullptr;
        int* stop = c.model ? nullptr : (int*)h->d_vstop.p;
        double* st = (double*)h->d_tpp_state.p;
        double* filt = (double*)h->d_tpp_filt.p;
        const int pgrid = (int)((n + 127) / 128);
        long long wblocks = (n + 3) / 4, wmax = (long long)h->num_sms * 16;
        const int wgrid = (int)(wblocks < wmax ? wblocks : wmax);
        CUDA_TRY(h, cudaEventRecord(h->ev0, s));
        for (int t = 0; t < c.T; t++) {
            rollout_plant_kernel<<<pgrid, 128, 0, s>>>((long long)n, Bp, veh, a.pose0, t == 0);
            if (c.model) rollout_frenet_ref_kernel<<<wgrid, 128, 0, s>>>(kc, fa, Bp, veh, fref);
            else rollout_waypoints_kernel<<<wgrid, 128, 0, s>>>(kc, (long long)n, Bp, veh, a.path_of, rg, st, filt, stop, t == 0);
            sk<<<(int)sblocks, tb, 0, s>>>(kc, (long long)n, Bp, veh, stop, st, filt, (!c.model && t == 0) ? a.warm0 : nullptr, des_speed, out,
                                           a.log ? a.log + (size_t)t * n * 8 : nullptr, fref, t == 0);
            if (a.met) rollout_metrics_kernel<<<wgrid, 128, 0, s>>>(kc, a, Bp, veh, stop, out.status, out.iters, t);
            CUDA_TRY(h, cudaGetLastError());
        }
        if (a.final_state) rollout_final_kernel<<<pgrid, 128, 0, s>>>((long long)n, Bp, veh, a.final_state);
        if (a.met) rollout_metrics_final_kernel<<<pgrid, 128, 0, s>>>((long long)n, Bp, a.met, (double*)h->d_metout.p);
        CUDA_TRY(h, cudaGetLastError());
        CUDA_TRY(h, cudaEventRecord(h->ev1, s));
        h->stats.kernel_launches += (a.met ? 4 : 3) * (int64_t)c.T + (a.final_state ? 1 : 0) + (a.met ? 1 : 0);
        return MPCB200_OK;
    }
    CUDA_TRY(h, cudaMemsetAsync(h->d_counter, 0, sizeof(unsigned long long), s));
    const int per_block = (h->team_warps == 1) ? WARPS_PER_BLOCK : 1;
    long long blocks_needed = (n + per_block - 1) / per_block;
    int bps = c.model ? h->frenet_rollout_blocks_per_sm : (c.w ? h->rollout_blocks_per_sm_w : h->rollout_blocks_per_sm);
    const int threads = 32 * (h->team_warps == 1 ? WARPS_PER_BLOCK : h->team_warps);
    const size_t smem = rollout_smem_bytes(h, c.w != nullptr);
    auto fk = c.metrics ? (c.w ? mpc_rollout_frenet_kernel<1, 1> : mpc_rollout_frenet_kernel<1, 0>)
                        : (c.w ? mpc_rollout_frenet_kernel<0, 1> : mpc_rollout_frenet_kernel<0, 0>);
    /* the MET = 1 and the Frenet PW = 1 instantiations: shared-memory limit and residency prepared here, by the calls that launch them */
    const void* prep_fn = nullptr;
    if (c.model && (c.metrics || c.w)) prep_fn = (const void*)fk;
    else if (!c.model && c.metrics) prep_fn = (const void*)(c.w ? rollout_kernel<1, 1>(h) : rollout_kernel<0, 1>(h));
    if (prep_fn) CUDA_TRY(h, prepare_kernel(prep_fn, h->device, threads, smem, &bps));
    long long max_blocks = (long long)h->num_sms * bps;
    const int grid = (int)(blocks_needed < max_blocks ? blocks_needed : max_blocks);
    CUDA_TRY(h, cudaEventRecord(h->ev0, s));
    if (c.model) fk<<<grid, threads, smem, s>>>(kc, fa, h->d_counter, a.met, a.w);
    else if (c.metrics) (c.w ? rollout_kernel<1, 1>(h) : rollout_kernel<0, 1>(h))<<<grid, threads, smem, s>>>(kc, a, h->d_counter);
    else (c.w ? rollout_kernel<1>(h) : rollout_kernel<0>(h))<<<grid, threads, smem, s>>>(kc, a, h->d_counter);
    if (c.metrics) rollout_metrics_final_kernel<<<(int)((n + 127) / 128), 128, 0, s>>>((long long)n, (long long)n, a.met, (double*)h->d_metout.p);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaEventRecord(h->ev1, s));
    h->stats.kernel_launches += c.metrics ? 2 : 1;
    return MPCB200_OK;
}

/* ... and copy the share's rows of log [T][B][8] (a strided block when the fleet is sliced) and final [B][8] back */
static int rollout_collect(mpcb200_handle* h, const RolloutCall& c, int64_t lo, int64_t n) {
    CUDA_TRY(h, cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const size_t row = (size_t)n * 8 * sizeof(double);
    if (c.log) {
        CUDA_TRY(h, cudaMemcpy2DAsync(c.log + (size_t)lo * 8, (size_t)c.B * 8 * sizeof(double), h->d_log.p, row, row, (size_t)c.T, cudaMemcpyDeviceToHost, s));
        h->stats.d2h_bytes += row * c.T;
    }
    if (c.final_state) { CUDA_TRY(h, cudaMemcpyAsync(c.final_state + (size_t)lo * 8, h->d_final.p, row, cudaMemcpyDeviceToHost, s)); h->stats.d2h_bytes += row; }
    if (c.metrics) {
        const size_t mrow = (size_t)n * MET_FIELDS * sizeof(double);
        CUDA_TRY(h, cudaMemcpyAsync(c.metrics + (size_t)lo * MET_FIELDS, h->d_metout.p, mrow, cudaMemcpyDeviceToHost, s));
        h->stats.d2h_bytes += mrow;
    }
    CUDA_TRY(h, cudaStreamSynchronize(s));
    float ms = 0.f;
    CUDA_TRY(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->stats.kernel_ms = ms;
    return MPCB200_OK;
}

/* the body of mpcb200_rollout, mpcb200_rollout_w (w == NULL: the handle's weights), mpcb200_rollout_frenet, mpcb200_rollout_frenet_w
 * and the _metrics forms */
static int rollout_impl(mpcb200_handle* h, const RolloutCall& c) {
    const char* who = c.who;
    if (!h) return MPCB200_EINVAL;
    if (c.B < 0 || c.T < 0) return fail(h, MPCB200_EINVAL, "%s: B=%lld T=%d", who, (long long)c.B, c.T);
    if (h->model != c.model)
        return fail(h, MPCB200_EINVAL, c.model ? "%s: the handle was not created with mpcb200_create_frenet" : "%s: not available for the Frenet-frame variant", who);
    if (c.model && h->team_warps != 1) return fail(h, MPCB200_EINVAL, "%s: N <= 31 (N=%d)", who, h->cfg.N);
    if (c.model && !(c.window >= 4.0 && c.window <= 500.0)) return fail(h, MPCB200_EINVAL, "%s: window %.3g m outside [4, 500]", who, c.window);
    memset(&h->stats, 0, sizeof(h->stats));
    if (c.B == 0 || c.T == 0) return MPCB200_OK;
    if (!c.pose0 || !c.path_of) return fail(h, MPCB200_EINVAL, "%s: pose0 and path_of are required", who);
    int rc;
    if ((rc = check_path_ids(h, who, "vehicle", c.B, c.path_of))) return rc;
    if (c.w && (rc = check_weight_rows(h, who, "vehicle", c.B, c.w, c.model ? 7 : 8))) return rc;
    /* a vehicle stays on one GPU for all T steps: contiguous slices of the fleet, every device at once.  Frenet fleets run on
     * devices[0] only, as mpc_b200.h documents */
    mpcb200_handle* dev[8];
    int64_t lo[8], hi[8];
    const int parts = slice_call(h, c.B, c.model ? 1 : h->n_sub + 1, dev, lo, hi);
    for (int i = 0; i < parts; i++)
        if ((rc = rollout_enqueue(dev[i], c, lo[i], hi[i] - lo[i]))) return sub_fail(h, dev[i], rc);
    for (int i = 0; i < parts; i++)
        if ((rc = rollout_collect(dev[i], c, lo[i], hi[i] - lo[i]))) return sub_fail(h, dev[i], rc);
    merge_stats(h, dev, parts);
    CUDA_TRY(h, cudaSetDevice(h->device));
    return MPCB200_OK;
}

int mpcb200_rollout(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of, int32_t track_using_time,
                    double target_vel, double* log, double* final_state) {
    return rollout_impl(h, {"mpcb200_rollout", 0, B, T, pose0, path_of, target_vel, track_using_time, nullptr, 0.0, 0, log, final_state, nullptr});
}

int mpcb200_rollout_w(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of, int32_t track_using_time,
                      double target_vel, const double* w, double* log, double* final_state) {
    if (h && !w && B > 0 && T > 0) return fail(h, MPCB200_EINVAL, "mpcb200_rollout_w: w is required");
    return rollout_impl(h, {"mpcb200_rollout_w", 0, B, T, pose0, path_of, target_vel, track_using_time, w, 0.0, 0, log, final_state, nullptr});
}

int mpcb200_rollout_frenet(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of, double window,
                           double target_vel, int32_t ey_from_path, double* log, double* final_state) {
    return rollout_impl(h, {"mpcb200_rollout_frenet", 1, B, T, pose0, path_of, target_vel, 0, nullptr, window, ey_from_path, log, final_state,
                            nullptr});
}

int mpcb200_rollout_frenet_w(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of, double window,
                             double target_vel, int32_t ey_from_path, const double* w, double* log, double* final_state, double* metrics) {
    if (h && !w && B > 0 && T > 0) return fail(h, MPCB200_EINVAL, "mpcb200_rollout_frenet_w: w is required");
    return rollout_impl(h, {"mpcb200_rollout_frenet_w", 1, B, T, pose0, path_of, target_vel, 0, w, window, ey_from_path, log, final_state,
                            metrics});
}

int mpcb200_rollout_metrics(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of, int32_t track_using_time,
                            double target_vel, const double* w, double* log, double* final_state, double* metrics) {
    if (h && !metrics) return fail(h, MPCB200_EINVAL, "mpcb200_rollout_metrics: metrics is required");
    return rollout_impl(h, {"mpcb200_rollout_metrics", 0, B, T, pose0, path_of, target_vel, track_using_time, w, 0.0, 0, log, final_state,
                            metrics});
}

int mpcb200_rollout_frenet_metrics(mpcb200_handle* h, int64_t B, int32_t T, const double* pose0, const int32_t* path_of, double window,
                                   double target_vel, int32_t ey_from_path, double* log, double* final_state, double* metrics) {
    if (h && !metrics) return fail(h, MPCB200_EINVAL, "mpcb200_rollout_frenet_metrics: metrics is required");
    return rollout_impl(h, {"mpcb200_rollout_frenet_metrics", 1, B, T, pose0, path_of, target_vel, 0, nullptr, window, ey_from_path, log,
                            final_state, metrics});
}

int mpcb200_get_stats(mpcb200_handle* h, mpcb200_stats* out) {
    if (!h || !out) return MPCB200_EINVAL;
    *out = h->stats;
    return MPCB200_OK;
}

int mpcb200_fp64_peak(mpcb200_handle* h, double* tflops) {
    if (!h || !tflops) return MPCB200_EINVAL;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const int threads = 256, blocks = h->num_sms * 8, iters = 1 << 15;
    double* d = nullptr;
    CUDA_TRY(h, cudaMalloc((void**)&d, (size_t)threads * blocks * sizeof(double)));
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        CUDA_TRY(h, cudaEventRecord(h->ev0, h->stream));
        fp64_peak_kernel<<<blocks, threads, 0, h->stream>>>(d, iters);
        CUDA_TRY(h, cudaEventRecord(h->ev1, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        float ms = 0.f;
        CUDA_TRY(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaFree(d);
    const double flops = 2.0 * 8.0 * (double)iters * threads * blocks;
    *tflops = flops / (best * 1e-3) / 1e12;
    return MPCB200_OK;
}

const char* mpcb200_last_error(mpcb200_handle* h) { return h ? h->err : g_err; }

}  // extern "C"
