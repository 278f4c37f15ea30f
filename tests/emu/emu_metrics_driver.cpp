// emu_metrics_driver.cpp -- TEST ONLY: the closed loops with tracking metrics (MET = 1) of the kernel sources on the CPU warp
// emulator.  It compiles emu_weights_driver.cpp (and with it emu_driver.cpp) as they stand and adds the metrics entry points.
#include "emu_weights_driver.cpp"

// metrics [B][MET_FIELDS] from the [MET_K][B] accumulators, as rollout_metrics_final_kernel does
static void finalize_all(long B, const std::vector<double>& met, double* metrics) {
    for (long v = 0; v < B; v++) metrics_finalize(met.data() + v, B, metrics + (size_t)MET_FIELDS * v);
}

// fused XY closed loop (rollout_group<W, PW, 1>, the source of mpc_rollout_kernel / mpc_rollout_long_kernel with MET = 1)
template <int PW> static void lane_rollout_met(int lane, void* p) {
    RJob* j = (RJob*)p;
    double* team = j->smem + (size_t)(lane >> 5) * j->per_team;
    TeamSolver<1, 0, PW>::init_work(team, j->cfg->N);
    rollout_group<1, PW, 1>(*j->cfg, *j->a, j->b0, team, j->smem + (size_t)4 * j->per_team, 4);
}
template <int W, int PW> static void lane_rollout_long_met(int, void* p) {
    RJob* j = (RJob*)p;
    TeamSolver<W, 0, PW>::init_work(j->smem, j->cfg->N);
    rollout_group<W, PW, 1>(*j->cfg, *j->a, j->b0, j->smem, j->smem + (size_t)j->per_team, 1);
}

// the pipeline's metrics kernel (rollout_metrics_kernel) for one vehicle and period: metrics_period on one warp
struct MJob { const KCfg* cfg; const PathTable* path; double* m; long stride; int t; double x, y, psi, acc, df; int status, iters; };
static void lane_metrics(int, void* p) {
    MJob* j = (MJob*)p;
    TeamSolver<1> S(*j->cfg, (smem_t) nullptr);
    metrics_period(S, j->m, j->stride, j->t, *j->path, j->x, j->y, j->psi, j->acc, j->df, j->status, j->iters);
}

// pw: the PW = 1 instantiation (w may then be null: KCfg::w through the per-vehicle path).  tpp: the per-period pipeline
// (plant, waypoints, thread-per-problem solve as emu_rollout_w mirrors them, then the metrics kernel), vehicle by vehicle
extern "C" int emu_rollout_metrics(const KCfg* cfg, long B, int T, const double* pose0, const int* path_of, int n0, const double* t,
                                   const double* X, const double* Y, const double* psi, const double* s, int track_using_time,
                                   double target_vel, const double* w, int pw, double* log, double* final_state, const double* warm0,
                                   int tpp, double* metrics) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<double> cb_store, met((size_t)MET_K * B, 0.0 / 0.0);
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
                int status_i = -1, iters_i = 0;
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
                    acc_des = u0[2 * v]; df_des = u0[2 * v + 1]; status_i = status[v]; iters_i = iters[v];
                    up_d = df_des; up_a = acc_des;
                } else { acc_des = -1.0; df_des = 0.0; }
                if (log) {
                    double* r = log + ((size_t)step * B + v) * 8;
                    r[0] = veh[0]; r[1] = veh[1]; r[2] = veh[2]; r[3] = veh[3]; r[4] = acc_des; r[5] = df_des; r[6] = status_i; r[7] = iters_i;
                }
                MJob mj{&kc, &path, met.data() + v, B, step, veh[0], veh[1], veh[2], acc_des, df_des, status_i, iters_i};
                emu::race_reset();
                emu::run_warp(lane_metrics, &mj, 1);
            }
            if (final_state) for (int i = 0; i < 8; i++) final_state[8 * v + i] = veh[i];
        }
        finalize_all(B, met, metrics);
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
    a.warm0 = warm0; a.w = w; a.met = met.data();
    const int per_team = smem_doubles_per_team(kc.N, 0, pw ? 1 : 0);
    std::vector<double> smem_raw((size_t)4 * per_team + 4 * ROLLOUT_PX + 2, 0.0);
    double* smem = smem_raw.data();
    if (((size_t)smem) & 15) smem++;
    const int per_run = (W > 1) ? 1 : 4;   // long horizons: one emulated block of W warps = one vehicle; else four warps = four vehicles
    void (*fn)(int, void*) = pw ? (W == 1 ? lane_rollout_met<1> : W == 2 ? lane_rollout_long_met<2, 1> : lane_rollout_long_met<3, 1>)
                                : (W == 1 ? lane_rollout_met<0> : W == 2 ? lane_rollout_long_met<2, 0> : lane_rollout_long_met<3, 0>);
    for (long b0 = 0; b0 < B; b0 += per_run) {
        RJob j{&kc, &a, b0, smem, per_team};
        emu::race_reset();
        for (int q = 0; q < (W > 1 ? 1 : 4); q++) register_benign(smem + (size_t)q * per_team, kc.N);
        emu::run_warp(fn, &j, W == 1 ? 4 : W);
    }
    finalize_all(B, met, metrics);
    return 0;
}

// fused Frenet closed loop (rollout_group_frenet<1>, the source of mpc_rollout_frenet_kernel<1>): one emulated block of four
// warps = four vehicles, one path table
struct FMJob { const KCfg* cfg; const FrenetRolloutArgs* a; long b0; double* smem; int per_team; double* met; };
static void lane_rollout_frenet_met(int lane, void* p) {
    FMJob* j = (FMJob*)p;
    double* team = j->smem + (size_t)(lane >> 5) * j->per_team;
    TeamSolver<1, 1>::init_work(team, j->cfg->N);
    rollout_group_frenet<1>(*j->cfg, *j->a, j->b0, team, j->smem + (size_t)4 * j->per_team, 4, j->met);
}
extern "C" int emu_rollout_frenet_metrics(const KCfg* cfg, long B, int T, const double* pose0, const int* path_of, int n0, const double* t,
                                          const double* X, const double* Y, const double* psi, const double* s, double window,
                                          double target_vel, int ey_from_path, double* log, double* final_state, double* metrics) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<int> roles(32 * ROLE_STRIDE_F);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, w_sd_of(1, 1), roles.data() + l * ROLE_STRIDE_F, 1);
    kc.roles = roles.data();
    int n1, n2;
    fit_grid_sizes(window, &n1, &n2);
    std::vector<double> P(4 * (size_t)(n1 + n2)), met((size_t)MET_K * B, 0.0 / 0.0);
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
        FMJob j{&kc, &a, b0, smem, per_team, met.data()};
        emu::race_reset();
        for (int q = 0; q < 4; q++) register_benign(smem + (size_t)q * per_team, kc.N, 1);
        emu::run_warp(lane_rollout_frenet_met, &j, 4);
    }
    finalize_all(B, met, metrics);
    return 0;
}
