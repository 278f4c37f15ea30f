// emu_frenet_driver.cpp -- TEST ONLY: the Frenet closed loop of the kernel sources on the CPU warp emulator, piece by piece.
// It compiles emu_driver.cpp as it stands and adds the reference of one control period (frenet_reference), the host helpers
// that size and build its fit matrices, the fused loop over three distinct path tables, and the per-period pipeline.
#include "emu_driver.cpp"

// the three path tables of a call: n[i] samples and the columns t, X, Y, psi, s of table i
struct Tables3 {
    const int* n; const double* const* t; const double* const* X; const double* const* Y; const double* const* psi; const double* const* s;
};

// FrenetRolloutArgs over three tables, with the host-built fit matrices of `window` (kept alive in P and cb_store)
static FrenetRolloutArgs frenet_args(const Tables3& tb, double window, std::vector<double>& P, std::vector<double> cb_store[3]) {
    int n1, n2;
    fit_grid_sizes(window, &n1, &n2);
    P.assign(4 * (size_t)(n1 + n2), 0.0);
    cubic_fit_matrix(n1, 0.5, P.data()); cubic_fit_matrix(n2, 0.25, P.data() + 4 * (size_t)n1);
    FrenetRolloutArgs a;
    memset(&a, 0, sizeof(a));
    for (int i = 0; i < 3; i++) a.paths[i] = make_path(tb.n[i], tb.t[i], tb.X[i], tb.Y[i], tb.psi[i], tb.s[i], cb_store[i]);
    a.P1 = P.data(); a.P2 = P.data() + 4 * (size_t)n1; a.n1 = n1; a.n2 = n2;
    return a;
}

extern "C" void emu_fit_grid_sizes(double window, int* n1, int* n2) { fit_grid_sizes(window, n1, n2); }
extern "C" void emu_cubic_fit_matrix(int n, double step, double* P) { cubic_fit_matrix(n, step, P); }

// frenet_reference on one emulated warp for one pose.  Lane 0 also records what the kernel samples (the nearest sample and
// the path ahead in the vehicle frame), computed with the functions frenet_reference calls.
struct RefJob { const KCfg* cfg; const FrenetRolloutArgs* a; const PathTable* path; double X, Y, yaw; double kc[4], ey, psi0;
                int bi; double* xw; double* yw; };
static void lane_frenet_reference(int lane, void* p) {
    RefJob* j = (RefJob*)p;
    TeamSolver<1, 1> S(*j->cfg, (smem_t) nullptr);   // (one-warp teams: collectives are shuffles only)
    double kc[4], ey, psi0;
    frenet_reference(S, *j->path, *j->a, j->X, j->Y, j->yaw, kc, ey, psi0);
    const PathTable& path = *j->path;
    const int bi = S.nearest_sample(path, j->X, j->Y);   // (a warp collective: every lane)
    if (lane != 0) return;
    for (int r = 0; r < 4; r++) j->kc[r] = kc[r];
    j->ey = ey; j->psi0 = psi0; j->bi = bi;
    double sps, cps;
    mpc_sincos(j->yaw, &sps, &cps);
    for (int g = 0; g < j->a->n1; g++) {
        const double sq = path.s[j->bi] + 0.5 * (double)g;
        const double dx = np_interp(sq, path.s, path.X, path.n) - j->X, dy = np_interp(sq, path.s, path.Y, path.n) - j->Y;
        j->xw[g] = cps * dx + sps * dy; j->yw[g] = -sps * dx + cps * dy;
    }
}
// M poses [M][3] on path table 0 of tb; out: kc [M][4], ey [M], psi0 [M], nearest sample [M], xw and yw [M][n1]
extern "C" int emu_frenet_reference(const KCfg* cfg, const Tables3* tb, double window, int ey_from_path, long M, const double* poses,
                                    double* kc, double* ey, double* psi0, int* bi, double* xw, double* yw) {
    KCfg kc_ = *cfg;
    kcfg_finalize(kc_);
    std::vector<double> P, cb_store[3];
    FrenetRolloutArgs a = frenet_args(*tb, window, P, cb_store);
    a.ey_from_path = ey_from_path;
    for (long m = 0; m < M; m++) {
        RefJob j;
        memset(&j, 0, sizeof(j));
        j.cfg = &kc_; j.a = &a; j.path = &a.paths[0]; j.X = poses[3 * m]; j.Y = poses[3 * m + 1]; j.yaw = poses[3 * m + 2];
        j.xw = xw + (size_t)m * a.n1; j.yw = yw + (size_t)m * a.n1;
        emu::race_reset();
        emu::run_warp(lane_frenet_reference, &j, 1);
        for (int r = 0; r < 4; r++) kc[4 * m + r] = j.kc[r];
        ey[m] = j.ey; psi0[m] = j.psi0; bi[m] = j.bi;
    }
    return 0;
}

// the fused closed loop (rollout_group_frenet, mpc_rollout_frenet_kernel's source): vehicle v on table path_of[v]; blocks of
// four warps = four vehicles, so a fleet whose size is not a multiple of four ends with a partly full block
extern "C" int emu_rollout_frenet3(const KCfg* cfg, long B, int T, const double* pose0, const int* path_of, const Tables3* tb,
                                   double window, double target_vel, int ey_from_path, double* log, double* final_state) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<int> roles(32 * ROLE_STRIDE_F);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, w_sd_of(1, 1), roles.data() + l * ROLE_STRIDE_F, 1);
    kc.roles = roles.data();
    std::vector<double> P, cb_store[3];
    FrenetRolloutArgs a = frenet_args(*tb, window, P, cb_store);
    a.pose0 = pose0; a.path_of = path_of;
    a.T = T; a.ey_from_path = ey_from_path; a.target_vel = target_vel; a.log = log; a.final_state = final_state; a.B = B;
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

// the per-period pipeline of mpcb200_rollout_frenet for large fleets (csrc/mpc_b200.cu: rollout_plant_kernel,
// rollout_frenet_ref_kernel, rollout_solve_tpp_kernel<1, 0>), vehicle by vehicle: the plant, frenet_reference on one warp, then
// the thread-per-problem Frenet solve from (0, e_y, -psi_start, v), all zeros in the first period and the previous solution after
extern "C" int emu_rollout_frenet_tpp(const KCfg* cfg, long B, int T, const double* pose0, const int* path_of, const Tables3* tb,
                                      double window, double target_vel, int ey_from_path, double* log, double* final_state) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<double> P, cb_store[3];
    FrenetRolloutArgs a = frenet_args(*tb, window, P, cb_store);
    a.ey_from_path = ey_from_path;
    const long S = 40;
    std::vector<double> st(tpp_state_doubles(kc.N, S, 1), 0.0 / 0.0), filt(tpp_filter_doubles(S), 0.0 / 0.0);
    std::vector<double> u0(2 * B), xw(a.n1), yw(a.n1);
    std::vector<int> status(B), iters(B);
    BatchPtrs out;
    memset(&out, 0, sizeof(out));
    out.u0 = u0.data(); out.status = status.data(); out.iters = iters.data();
    for (long v = 0; v < B; v++) {
        const TppMemT<1> m(st.data(), filt.data(), kc.N, v % S);
        double veh[8] = {pose0[3 * v], pose0[3 * v + 1], pose0[3 * v + 2], 0, 0, 0, 0, 0};
        double acc_des = 0.0, df_des = 0.0, up_d = 0.0, up_a = 0.0;
        for (int step = 0; step < T; step++) {
            for (int i = 0; i < 10; i++) plant_step(veh, acc_des, df_des);
            RefJob j;
            memset(&j, 0, sizeof(j));
            j.cfg = &kc; j.a = &a; j.path = &a.paths[path_of[v]]; j.X = veh[0]; j.Y = veh[1]; j.yaw = veh[2];
            j.xw = xw.data(); j.yw = yw.data();
            emu::race_reset();
            emu::run_warp(lane_frenet_reference, &j, 1);
            TppSolverT<1> sv(kc, m);
            for (int i = 0; i < 4; i++) sv.kp[i] = j.kc[i];
            const double c7[7] = {0.0, j.ey, -j.psi0, veh[3], up_d, up_a, target_vel};
            if (step == 0) {   // start = 0.0, then the previous solution
                for (int k = 0; k <= kc.N; k++) for (int f = TF_SX; f <= TF_UD; f++) m.sto(f, k, 0.0);
                for (int k = 0; k <= kc.N; k++) { m.sto(TF_XR, k, 0.0); m.sto(TF_YR, k, 0.0); m.sto(TF_PR, k, 0.0); }
            }
            sv.begin_in_place(c7, nullptr);
            while (!sv.tick(true)) {}
            sv.finish(out, v);
            acc_des = u0[2 * v]; df_des = u0[2 * v + 1];   // published whatever the status
            up_d = df_des; up_a = acc_des;                 // update_current_input(df_opt, a_opt)
            if (log) {
                double* r = log + ((size_t)step * B + v) * 8;
                r[0] = veh[0]; r[1] = veh[1]; r[2] = veh[2]; r[3] = veh[3]; r[4] = acc_des; r[5] = df_des; r[6] = status[v]; r[7] = iters[v];
            }
        }
        if (final_state) for (int i = 0; i < 8; i++) final_state[8 * v + i] = veh[i];
    }
    return 0;
}
