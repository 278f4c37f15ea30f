// emu_driver.cpp -- TEST ONLY: runs mpc_kernel.cuh on the CPU warp emulator.
#define MPC_HOST_EMU 1
#include "warp_emu.h"
#include "mpc_kernel.cuh"

#include <vector>

namespace mpcb200 { namespace emu {
thread_local Warp* W = nullptr;
thread_local RaceState RS;

static void trampoline(int lane) {
    Warp* w = W;
    w->fn(lane, w->arg);
    w->done[lane] = 1;
    // hand over to the next unfinished lane, or back to main when all are done
    for (int i = 1; i <= w->nl; i++) {
        int c = (lane + i) % w->nl;
        if (!w->done[c]) { w->cur = c; setcontext(&w->ctx[c]); }
    }
    setcontext(&w->main_ctx);
}

void run_warp(void (*fn)(int, void*), void* arg, int warps) {
    static thread_local Warp w;
    memset(&w, 0, sizeof(w));
    const size_t STK = 1 << 18;
    w.nl = 32 * warps;
    w.stacks = (char*)malloc(w.nl * STK);
    w.fn = fn; w.arg = arg;
    W = &w;
    for (int l = 0; l < w.nl; l++) {
        getcontext(&w.ctx[l]);
        w.ctx[l].uc_stack.ss_sp = w.stacks + l * STK;
        w.ctx[l].uc_stack.ss_size = STK;
        w.ctx[l].uc_link = &w.main_ctx;
        makecontext(&w.ctx[l], (void (*)())trampoline, 1, l);
    }
    w.cur = 0;
    swapcontext(&w.main_ctx, &w.ctx[0]);
    free(w.stacks);
    W = nullptr;
}
}}  // namespace

using namespace mpcb200;

// PathTable over the caller's columns, with the chunk bounds mpcb200_set_path computes (kept alive in `store`)
static PathTable make_path(int n0, const double* t, const double* X, const double* Y, const double* psi, const double* s, std::vector<double>& store) {
    PathTable p;
    p.n = n0; p.t = t; p.X = X; p.Y = Y; p.psi = psi; p.s = s;
    p.nch = path_chunks(n0);
    store.resize((size_t)3 * p.nch);
    path_chunk_bounds(n0, X, Y, store.data());
    p.cb = store.data();
    return p;
}


// benign words of one team's shared memory: the sink of inactive lanes and, in every per-thread
// state group, the slot shared by the threads that own no stage
static void register_benign(double* team, int N, int model = 0) {
    emu::race_benign(team + W_DUMMY, 1, 2);
    const int go[6] = {G_EV_OFF, G_REF_OFF, G_DX_OFF, G_DRS_OFF, G_DY_OFF, G_Z_OFF};
    const int gs[6] = {G_EV_STRIDE, model ? 4 : G_REF_STRIDE, G_DX_STRIDE, G_DRS_STRIDE, G_DY_STRIDE, G_Z_STRIDE};
    for (int g = 0; g < 6; g++) emu::race_benign(team + lf_offset(N, model) + go[g] * (N + 2) + gs[g] * (N + 1), 1, gs[g]);
}
extern "C" long emu_race_count() { return emu::RS.races; }
extern "C" void emu_race_enable(int on) { emu::RS.enabled = on; emu::RS.races = 0; }

struct Job { const KCfg* cfg; const BatchPtrs* io; long b; double* smem; };
template <int W> static void lane_main(int, void* a) {
    Job* j = (Job*)a;
    TeamSolver<W>::init_work(j->smem, j->cfg->N);
    RefGen rg;
    memset(&rg, 0, sizeof(rg));
    solve_problem<W>(*j->cfg, *j->io, rg, j->b, j->smem);
}

extern "C" int emu_solve_batch(const KCfg* cfg, long B, const double* state, const double* ref, const double* v_des,
                               const double* u_prev, double* warm, double* u0, double* cost, int* status, int* iters,
                               double* traj) {
    BatchPtrs io{state, ref, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, nullptr};
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<int> roles(32 * ROLE_STRIDE + 32 * RS_STRIDE);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, W_SD_OF(team_warps(kc.N)), roles.data() + l * ROLE_STRIDE);
    for (int l = 0; l < 32; l++) riccati_roles_shfl(l, kc.N, W_SD_OF(team_warps(kc.N)), roles.data() + 32 * ROLE_STRIDE + l * RS_STRIDE);
    kc.roles = roles.data();
    std::vector<double> smem_raw(smem_doubles_per_team(kc.N) + 2, 0.0);
    double* smem = smem_raw.data();
    if (((size_t)smem) & 15) smem++;   // 16-byte alignment like the device's shared memory
    const int W = team_warps(kc.N);
    for (long b = 0; b < B; b++) {
        Job j{&kc, &io, b, smem};
        emu::race_reset();
        register_benign(smem, kc.N);
        emu::run_warp(W == 1 ? lane_main<1> : W == 2 ? lane_main<2> : lane_main<3>, &j, W);
    }
    return 0;
}
template <int W> static void lane_main_frenet(int, void* a) {
    Job* j = (Job*)a;
    TeamSolver<W, 1>::init_work(j->smem, j->cfg->N);
    RefGen rg;
    memset(&rg, 0, sizeof(rg));
    solve_problem<W, 1>(*j->cfg, *j->io, rg, j->b, j->smem);
}
// Frenet-frame variant: ref = [B][4] curvature polynomial
extern "C" int emu_solve_batch_frenet(const KCfg* cfg, long B, const double* state, const double* kpoly, const double* v_des,
                                      const double* u_prev, double* warm, double* u0, double* cost, int* status, int* iters,
                                      double* traj) {
    BatchPtrs io{state, kpoly, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, nullptr};
    KCfg kc = *cfg;
    if (kc.N > 95) return -1;
    kcfg_finalize(kc);
    const int W = team_warps(kc.N);
    std::vector<int> roles(32 * ROLE_STRIDE_F);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, w_sd_of(W, 1), roles.data() + l * ROLE_STRIDE_F, 1);
    kc.roles = roles.data();
    std::vector<double> smem_raw(smem_doubles_per_team(kc.N, 1) + 2, 0.0);
    double* smem = smem_raw.data();
    if (((size_t)smem) & 15) smem++;
    for (long b = 0; b < B; b++) {
        Job j{&kc, &io, b, smem};
        emu::race_reset();
        register_benign(smem, kc.N, 1);
        emu::run_warp(W == 1 ? lane_main_frenet<1> : W == 2 ? lane_main_frenet<2> : lane_main_frenet<3>, &j, W);
    }
    return 0;
}
extern "C" int emu_kcfg_size() { return (int)sizeof(KCfg); }

struct RJob { const KCfg* cfg; const RolloutArgs* a; long b0; double* smem; int per_team; };
static void lane_rollout(int lane, void* p) {
    RJob* j = (RJob*)p;
    double* team = j->smem + (size_t)(lane >> 5) * j->per_team;
    TeamSolver<1>::init_work(team, j->cfg->N);
    rollout_group<1>(*j->cfg, *j->a, j->b0, team, j->smem + (size_t)4 * j->per_team, 4);
}
template <int W> static void lane_rollout_long(int, void* p) {
    RJob* j = (RJob*)p;
    TeamSolver<W>::init_work(j->smem, j->cfg->N);
    rollout_group<W>(*j->cfg, *j->a, j->b0, j->smem, j->smem + (size_t)j->per_team, 1);
}
// warm0: [6N+4] start point of every vehicle's first solve, or null (all zeros)
extern "C" int emu_rollout(const KCfg* cfg, long B, int T, const double* pose0, const int* path_of, int n0, const double* t,
                           const double* X, const double* Y, const double* psi, const double* s, int track_using_time,
                           double target_vel, double* log, double* final_state, const double* warm0) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    const int W = team_warps(kc.N);
    std::vector<int> roles(32 * ROLE_STRIDE + 32 * RS_STRIDE);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, W_SD_OF(W), roles.data() + l * ROLE_STRIDE);
    for (int l = 0; l < 32; l++) riccati_roles_shfl(l, kc.N, W_SD_OF(W), roles.data() + 32 * ROLE_STRIDE + l * RS_STRIDE);
    kc.roles = roles.data();
    RolloutArgs a;
    memset(&a, 0, sizeof(a));
    a.pose0 = pose0; a.path_of = path_of;
    std::vector<double> cb_store;
    for (int i = 0; i < 3; i++) a.paths[i] = make_path(n0, t, X, Y, psi, s, cb_store);
    a.T = T; a.track_using_time = track_using_time; a.target_vel = target_vel; a.log = log; a.final_state = final_state; a.B = B;
    a.warm0 = warm0;
    const int per_team = smem_doubles_per_team(kc.N);
    std::vector<double> smem_raw((size_t)4 * per_team + 4 * ROLLOUT_PX + 2, 0.0);
    double* smem = smem_raw.data();
    if (((size_t)smem) & 15) smem++;
    if (W > 1) {   // long horizons: one emulated block of W warps = one vehicle
        for (long b0 = 0; b0 < B; b0++) {
            RJob j{&kc, &a, b0, smem, per_team};
            emu::race_reset();
            register_benign(smem, kc.N);
            emu::run_warp(W == 2 ? lane_rollout_long<2> : lane_rollout_long<3>, &j, W);
        }
        return 0;
    }
    for (long b0 = 0; b0 < B; b0 += 4) {   // one emulated block of four warps = four vehicles
        RJob j{&kc, &a, b0, smem, per_team};
        emu::race_reset();
        for (int w = 0; w < 4; w++) register_benign(smem + (size_t)w * per_team, kc.N);
        emu::run_warp(lane_rollout, &j, 4);
    }
    return 0;
}

// open-loop batch with the waypoints generated by the kernel from one path table (mpcb200_solve_batch_on_path)
struct PJob { const KCfg* cfg; const BatchPtrs* io; const RefGen* rg; long b; double* smem; };
template <int W> static void lane_on_path(int, void* p) {
    PJob* j = (PJob*)p;
    TeamSolver<W>::init_work(j->smem, j->cfg->N);
    solve_problem<W>(*j->cfg, *j->io, *j->rg, j->b, j->smem);
}
extern "C" int emu_solve_batch_on_path(const KCfg* cfg, long B, const double* state, const int* path_of, int n0, const double* t,
                                       const double* X, const double* Y, const double* psi, const double* s, int track_using_time,
                                       double target_vel, const double* u_prev, double* u0, double* cost, int* status, int* iters,
                                       double* traj, double* ref_out, int* stop) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    const int W = team_warps(kc.N);
    std::vector<int> roles(32 * ROLE_STRIDE + 32 * RS_STRIDE);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, W_SD_OF(W), roles.data() + l * ROLE_STRIDE);
    for (int l = 0; l < 32; l++) riccati_roles_shfl(l, kc.N, W_SD_OF(W), roles.data() + 32 * ROLE_STRIDE + l * RS_STRIDE);
    kc.roles = roles.data();
    BatchPtrs io{state, nullptr, nullptr, u_prev, nullptr, u0, cost, status, iters, traj, nullptr, nullptr};
    RefGen rg;
    memset(&rg, 0, sizeof(rg));
    rg.path_of = path_of;
    std::vector<double> cb_store;
    rg.paths[0] = make_path(n0, t, X, Y, psi, s, cb_store);
    rg.track_using_time = track_using_time; rg.target_vel = target_vel > 0.0 ? target_vel : 0.0; rg.ref_out = ref_out; rg.stop = stop;
    std::vector<double> smem_raw(smem_doubles_per_team(kc.N) + 2, 0.0);
    double* smem = smem_raw.data();
    if (((size_t)smem) & 15) smem++;
    for (long b = 0; b < B; b++) {
        PJob j{&kc, &io, &rg, b, smem};
        emu::race_reset();
        register_benign(smem, kc.N);
        emu::run_warp(W == 1 ? lane_on_path<1> : W == 2 ? lane_on_path<2> : lane_on_path<3>, &j, W);
    }
    return 0;
}

// closed loop on the Frenet-frame module (rollout_group_frenet): one emulated block of four warps = four vehicles
struct FJob { const KCfg* cfg; const FrenetRolloutArgs* a; long b0; double* smem; int per_team; };
static void lane_rollout_frenet(int lane, void* p) {
    FJob* j = (FJob*)p;
    double* team = j->smem + (size_t)(lane >> 5) * j->per_team;
    TeamSolver<1, 1>::init_work(team, j->cfg->N);
    rollout_group_frenet(*j->cfg, *j->a, j->b0, team, j->smem + (size_t)4 * j->per_team, 4);
}
extern "C" int emu_rollout_frenet(const KCfg* cfg, long B, int T, const double* pose0, const int* path_of, int n0, const double* t,
                                  const double* X, const double* Y, const double* psi, const double* s, double window,
                                  double target_vel, int ey_from_path, double* log, double* final_state) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<int> roles(32 * ROLE_STRIDE_F);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, w_sd_of(1, 1), roles.data() + l * ROLE_STRIDE_F, 1);
    kc.roles = roles.data();
    int n1, n2;
    fit_grid_sizes(window, &n1, &n2);
    std::vector<double> P(4 * (size_t)(n1 + n2));
    cubic_fit_matrix(n1, 0.5, P.data()); cubic_fit_matrix(n2, 0.25, P.data() + 4 * (size_t)n1);
    FrenetRolloutArgs a;
    memset(&a, 0, sizeof(a));
    a.pose0 = pose0; a.path_of = path_of;
    std::vector<double> cb_store;
    for (int i = 0; i < 3; i++) a.paths[i] = make_path(n0, t, X, Y, psi, s, cb_store);
    a.T = T; a.ey_from_path = ey_from_path; a.target_vel = target_vel; a.log = log; a.final_state = final_state; a.B = B;
    a.P1 = P.data(); a.P2 = P.data() + 4 * (size_t)n1; a.n1 = n1; a.n2 = n2;
    const int per_team = smem_doubles_per_team(kc.N, 1);
    std::vector<double> smem_raw((size_t)4 * per_team + 4 * ROLLOUT_PX + 2, 0.0);
    double* smem = smem_raw.data();
    if (((size_t)smem) & 15) smem++;
    for (long b0 = 0; b0 < B; b0 += 4) {
        FJob j{&kc, &a, b0, smem, per_team};
        emu::race_reset();
        for (int w = 0; w < 4; w++) register_benign(smem + (size_t)w * per_team, kc.N, 1);
        emu::run_warp(lane_rollout_frenet, &j, 4);
    }
    return 0;
}

// ---- thread-per-problem solver (csrc/tpp_solver.cuh): plain scalar code, no emulated warp needed.  The problems go
// round-robin over S slots of one state array, so the [field][stage][slot] addressing of the device layout is exercised.
#include "tpp_solver.cuh"
extern "C" int emu_solve_batch_tpp(const KCfg* cfg, long B, const double* state, const double* ref, const double* v_des,
                                   const double* u_prev, double* warm, double* u0, double* cost, int* status, int* iters,
                                   double* traj, int* resto, long S, long* ticks) {
    BatchPtrs io{state, ref, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, resto};
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    if (S < 1) S = 1;
    std::vector<double> st(tpp_state_doubles(kc.N, S), 0.0 / 0.0), filt(tpp_filter_doubles(S), 0.0 / 0.0);   // NaN: a field read before it is written shows
    for (long b = 0; b < B; b++) {
        TppMem m(st.data(), filt.data(), kc.N, b % S);
        TppSolver sv(kc, m);
        sv.begin(io, b);
        long t = 0;
        while (!sv.tick(true)) t++;
        if (ticks) ticks[b] = t;
        sv.finish(io, b);
    }
    return 0;
}

// closed loop with the thread-per-problem solve, as mpcb200_rollout runs it for large fleets (plant / waypoints / solve per
// control period; csrc/mpc_b200.cu: rollout_plant_kernel, rollout_waypoints_kernel, rollout_solve_tpp_kernel), vehicle by vehicle
struct WJob { const KCfg* cfg; const PathTable* path; double X, Y, yaw; int use_vt; double vt; TppMem* mem; int stop; };
static void lane_waypoints(int lane, void* p) {
    WJob* j = (WJob*)p;
    TeamSolver<1> S(*j->cfg, (smem_t) nullptr);
    double xr, yr, pr;
    const bool sc = S.get_waypoints(*j->path, j->cfg->dt, j->X, j->Y, j->yaw, j->use_vt != 0, j->vt, xr, yr, pr);
    if (lane <= j->cfg->N) { j->mem->sto(TF_XR, lane, xr); j->mem->sto(TF_YR, lane, yr); j->mem->sto(TF_PR, lane, pr); }
    if (sc && lane == 0) j->stop = 1;
}
extern "C" int emu_rollout_tpp(const KCfg* cfg, long B, int T, const double* pose0, const int* path_of, int n0, const double* t,
                               const double* X, const double* Y, const double* psi, const double* s, int track_using_time,
                               double target_vel, double* log, double* final_state, const double* warm0) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<double> cb_store;
    PathTable path = make_path(n0, t, X, Y, psi, s, cb_store);
    (void)path_of;   // (the emulator gets one path table, like emu_rollout)
    const double des_speed = target_vel > 0.0 ? target_vel : 0.0;
    const long S = 40;
    std::vector<double> st(tpp_state_doubles(kc.N, S), 0.0 / 0.0), filt(tpp_filter_doubles(S), 0.0 / 0.0);
    std::vector<double> u0(2 * B); std::vector<int> status(B), iters(B);
    BatchPtrs out;
    memset(&out, 0, sizeof(out));
    out.u0 = u0.data(); out.status = status.data(); out.iters = iters.data();
    for (long v = 0; v < B; v++) {
        TppMem m(st.data(), filt.data(), kc.N, v % S);
        double veh[8] = {pose0[3 * v], pose0[3 * v + 1], pose0[3 * v + 2], 0, 0, 0, 0, 0};
        double acc_des = 0.0, df_des = 0.0, up_d = 0.0, up_a = 0.0;
        int stop = 0;
        for (int step = 0; step < T; step++) {
            for (int i = 0; i < 10; i++) plant_step(veh, acc_des, df_des);
            double status_f = -1.0, iters_f = 0.0;
            if (!stop) {
                WJob j{&kc, &path, veh[0], veh[1], veh[2], !track_using_time, des_speed, &m, 0};
                emu::race_reset();
                emu::run_warp(lane_waypoints, &j, 1);
                stop = j.stop;
            }
            if (!stop) {
                TppSolver sv(kc, m);
                const double c7[7] = {veh[0], veh[1], veh[2], veh[3], up_d, up_a, des_speed};
                sv.begin_in_place(c7, step == 0 ? warm0 : nullptr);
                while (!sv.tick(true)) {}
                sv.finish(out, v);
                acc_des = u0[2 * v]; df_des = u0[2 * v + 1]; status_f = status[v]; iters_f = iters[v];
                up_d = df_des; up_a = acc_des;
            } else { acc_des = -1.0; df_des = 0.0; }
            if (log) {
                double* r = log + ((size_t)step * B + v) * 8;
                r[0] = veh[0]; r[1] = veh[1]; r[2] = veh[2]; r[3] = veh[3]; r[4] = acc_des; r[5] = df_des; r[6] = status_f; r[7] = iters_f;
            }
        }
        if (final_state) for (int i = 0; i < 8; i++) final_state[8 * v + i] = veh[i];
    }
    return 0;
}

// thread-per-problem solver, Frenet-frame variant (MODEL 1): ref = [B][4] curvature polynomial
extern "C" int emu_solve_batch_tpp_frenet(const KCfg* cfg, long B, const double* state, const double* kpoly, const double* v_des,
                                          const double* u_prev, double* warm, double* u0, double* cost, int* status, int* iters,
                                          double* traj, int* resto, long S) {
    BatchPtrs io{state, kpoly, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, resto};
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    if (S < 1) S = 1;
    std::vector<double> st(tpp_state_doubles(kc.N, S, 1), 0.0 / 0.0), filt(tpp_filter_doubles(S), 0.0 / 0.0);
    for (long b = 0; b < B; b++) {
        TppMemT<1> m(st.data(), filt.data(), kc.N, b % S);
        TppSolverT<1> sv(kc, m);
        sv.begin(io, b);
        while (!sv.tick(true)) {}
        sv.finish(io, b);
    }
    return 0;
}
