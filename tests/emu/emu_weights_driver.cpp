// emu_weights_driver.cpp -- TEST ONLY: the per-problem-weight (PW = 1) instantiations of the kernel sources on the CPU warp
// emulator.  It compiles emu_driver.cpp as it stands and adds the weighted entry points, so both share one emulator.
#include "emu_driver.cpp"

// ---- per-problem cost weights (mpcb200_solve_batch_w / _frenet_w / mpcb200_rollout_w): the PW = 1 instantiations of the same
// sources.  w = [B][8] ([B][7] Frenet) or null (KCfg::w, through the per-problem path).  Bad rows are not checked here: the kernels
// answer them (MPCB200_ERROR), as they do for device pointers.
template <int W, int MODEL> static void lane_main_w(int, void* a) {
    Job* j = (Job*)a;
    TeamSolver<W, MODEL, 1>::init_work(j->smem, j->cfg->N);
    RefGen rg;
    memset(&rg, 0, sizeof(rg));
    solve_problem<W, MODEL, 1>(*j->cfg, *j->io, rg, j->b, j->smem);
}
template <int MODEL>
static int solve_batch_w(const KCfg* cfg, long B, const BatchPtrs& io) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    const int W = team_warps(kc.N);
    const int rs = role_stride_of(MODEL);
    std::vector<int> roles(32 * rs + 32 * RS_STRIDE);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, w_sd_of(W, MODEL), roles.data() + l * rs, MODEL);
    for (int l = 0; l < 32; l++) riccati_roles_shfl(l, kc.N, w_sd_of(W, MODEL), roles.data() + 32 * rs + l * RS_STRIDE);
    kc.roles = roles.data();
    std::vector<double> smem_raw(smem_doubles_per_team(kc.N, MODEL, 1) + 2, 0.0);
    double* smem = smem_raw.data();
    if (((size_t)smem) & 15) smem++;
    for (long b = 0; b < B; b++) {
        Job j{&kc, &io, b, smem};
        emu::race_reset();
        register_benign(smem, kc.N, MODEL);
        emu::run_warp(W == 1 ? lane_main_w<1, MODEL> : W == 2 ? lane_main_w<2, MODEL> : lane_main_w<3, MODEL>, &j, W);
    }
    return 0;
}
template <int MODEL>
static int solve_batch_tpp_w(const KCfg* cfg, long B, const BatchPtrs& io, long S) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    if (S < 1) S = 1;
    std::vector<double> st(tpp_state_doubles(kc.N, S, MODEL), 0.0 / 0.0), filt(tpp_filter_doubles(S), 0.0 / 0.0);
    for (long b = 0; b < B; b++) {
        if (io.w && !row_weights_ok(io.w, b, MODEL)) { write_error_answer(io, b); continue; }   // as mpc_solve_tpp_kernel does
        TppMemT<MODEL> m(st.data(), filt.data(), kc.N, b % S);
        TppSolverT<MODEL, 1> sv(kc, m);
        sv.begin(io, b);
        while (!sv.tick(true)) {}
        sv.finish(io, b);
    }
    return 0;
}
extern "C" int emu_solve_batch_w(const KCfg* cfg, long B, const double* state, const double* ref, const double* v_des, const double* u_prev,
                                 double* warm, const double* w, double* u0, double* cost, int* status, int* iters, double* traj, int* resto) {
    const BatchPtrs io{state, ref, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, resto, w};
    return solve_batch_w<0>(cfg, B, io);
}
extern "C" int emu_solve_batch_frenet_w(const KCfg* cfg, long B, const double* state, const double* kpoly, const double* v_des,
                                        const double* u_prev, double* warm, const double* w, double* u0, double* cost, int* status,
                                        int* iters, double* traj, int* resto) {
    const BatchPtrs io{state, kpoly, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, resto, w};
    return solve_batch_w<1>(cfg, B, io);
}
extern "C" int emu_solve_batch_tpp_w(const KCfg* cfg, long B, const double* state, const double* ref, const double* v_des, const double* u_prev,
                                     double* warm, const double* w, double* u0, double* cost, int* status, int* iters, double* traj, int* resto,
                                     long S) {
    const BatchPtrs io{state, ref, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, resto, w};
    return solve_batch_tpp_w<0>(cfg, B, io, S);
}
extern "C" int emu_solve_batch_tpp_frenet_w(const KCfg* cfg, long B, const double* state, const double* kpoly, const double* v_des,
                                            const double* u_prev, double* warm, const double* w, double* u0, double* cost, int* status,
                                            int* iters, double* traj, int* resto, long S) {
    const BatchPtrs io{state, kpoly, v_des, u_prev, warm, u0, cost, status, iters, traj, nullptr, resto, w};
    return solve_batch_tpp_w<1>(cfg, B, io, S);
}

// closed loop with per-vehicle weights: the fused kernel's source (rollout_group<W, 1>) or, tpp != 0, the per-period pipeline
// (rollout_solve_tpp_kernel<0, 1>: the slot's solver reads its vehicle's row)
static void lane_rollout_w(int lane, void* p) {
    RJob* j = (RJob*)p;
    double* team = j->smem + (size_t)(lane >> 5) * j->per_team;
    TeamSolver<1, 0, 1>::init_work(team, j->cfg->N);
    rollout_group<1, 1>(*j->cfg, *j->a, j->b0, team, j->smem + (size_t)4 * j->per_team, 4);
}
template <int W> static void lane_rollout_long_w(int, void* p) {
    RJob* j = (RJob*)p;
    TeamSolver<W, 0, 1>::init_work(j->smem, j->cfg->N);
    rollout_group<W, 1>(*j->cfg, *j->a, j->b0, j->smem, j->smem + (size_t)j->per_team, 1);
}
extern "C" int emu_rollout_w(const KCfg* cfg, long B, int T, const double* pose0, const int* path_of, int n0, const double* t,
                             const double* X, const double* Y, const double* psi, const double* s, int track_using_time,
                             double target_vel, const double* w, double* log, double* final_state, const double* warm0, int tpp) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<double> cb_store;
    if (tpp) {
        PathTable path = make_path(n0, t, X, Y, psi, s, cb_store);
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
                    TppSolverT<0, 1> sv(kc, m);
                    sv.wr = w ? w + 8 * v : nullptr;
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
    const int W = team_warps(kc.N);
    std::vector<int> roles(32 * ROLE_STRIDE + 32 * RS_STRIDE);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, W_SD_OF(W), roles.data() + l * ROLE_STRIDE);
    for (int l = 0; l < 32; l++) riccati_roles_shfl(l, kc.N, W_SD_OF(W), roles.data() + 32 * ROLE_STRIDE + l * RS_STRIDE);
    kc.roles = roles.data();
    RolloutArgs a;
    memset(&a, 0, sizeof(a));
    a.pose0 = pose0; a.path_of = path_of;
    for (int i = 0; i < 3; i++) a.paths[i] = make_path(n0, t, X, Y, psi, s, cb_store);
    a.T = T; a.track_using_time = track_using_time; a.target_vel = target_vel; a.log = log; a.final_state = final_state; a.B = B;
    a.warm0 = warm0; a.w = w;
    const int per_team = smem_doubles_per_team(kc.N, 0, 1);
    std::vector<double> smem_raw((size_t)4 * per_team + 4 * ROLLOUT_PX + 2, 0.0);
    double* smem = smem_raw.data();
    if (((size_t)smem) & 15) smem++;
    const int per_run = (W > 1) ? 1 : 4;   // long horizons: one emulated block of W warps = one vehicle; else four warps = four vehicles
    for (long b0 = 0; b0 < B; b0 += per_run) {
        RJob j{&kc, &a, b0, smem, per_team};
        emu::race_reset();
        for (int q = 0; q < (W > 1 ? 1 : 4); q++) register_benign(smem + (size_t)q * per_team, kc.N);
        emu::run_warp(W == 1 ? lane_rollout_w : W == 2 ? lane_rollout_long_w<2> : lane_rollout_long_w<3>, &j, W == 1 ? 4 : W);
    }
    return 0;
}
