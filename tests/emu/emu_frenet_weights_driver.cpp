// emu_frenet_weights_driver.cpp -- TEST ONLY: the Frenet closed loop with per-vehicle cost weights (mpcb200_rollout_frenet_w) of the
// kernel sources on the CPU warp emulator.  It compiles emu_frenet_driver.cpp (and with it emu_driver.cpp) as they stand and adds
// the PW = 1 forms of its fused loop and its per-period pipeline.
#include "emu_frenet_driver.cpp"

// fused closed loop (rollout_group_frenet<MET, 1>, the source of mpc_rollout_frenet_kernel<MET, 1>): blocks of four warps = four
// vehicles, each staging its own row [B][7]
struct FWJob { const KCfg* cfg; const FrenetRolloutArgs* a; long b0; double* smem; int per_team; double* met; const double* w; };
template <int MET> static void lane_rollout_frenet_w(int lane, void* p) {
    FWJob* j = (FWJob*)p;
    double* team = j->smem + (size_t)(lane >> 5) * j->per_team;
    TeamSolver<1, 1, 1>::init_work(team, j->cfg->N);
    rollout_group_frenet<MET, 1>(*j->cfg, *j->a, j->b0, team, j->smem + (size_t)4 * j->per_team, 4, j->met, j->w);
}

// w [B][7] (cey, cep, cev, cda, cdd, ca, cd); metrics [B][MET_FIELDS] or null (MET = 0).  tpp: the per-period pipeline as
// emu_rollout_frenet_tpp runs it, with the slot's TppSolverT<1, 1> reading its vehicle's row (rollout_solve_tpp_kernel<1, 1>);
// that form has no metrics here (its metrics kernel is the unweighted pipeline's).
extern "C" int emu_rollout_frenet_w(const KCfg* cfg, long B, int T, const double* pose0, const int* path_of, const Tables3* tb,
                                    double window, double target_vel, int ey_from_path, const double* w, double* log,
                                    double* final_state, double* metrics, int tpp) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<double> P, cb_store[3];
    FrenetRolloutArgs a = frenet_args(*tb, window, P, cb_store);
    a.ey_from_path = ey_from_path;
    if (tpp) {
        if (metrics) return -1;
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
                TppSolverT<1, 1> sv(kc, m);
                sv.wr = w + 7 * v;
                for (int i = 0; i < 4; i++) sv.kp[i] = j.kc[i];
                const double c7[7] = {0.0, j.ey, -j.psi0, veh[3], up_d, up_a, target_vel};
                if (step == 0) {   // start = 0.0, then the previous solution
                    for (int k = 0; k <= kc.N; k++) for (int f = TF_SX; f <= TF_UD; f++) m.sto(f, k, 0.0);
                    for (int k = 0; k <= kc.N; k++) { m.sto(TF_XR, k, 0.0); m.sto(TF_YR, k, 0.0); m.sto(TF_PR, k, 0.0); }
                }
                sv.begin_in_place(c7, nullptr);
                while (!sv.tick(true)) {}
                sv.finish(out, v);
                acc_des = u0[2 * v]; df_des = u0[2 * v + 1];
                up_d = df_des; up_a = acc_des;
                if (log) {
                    double* r = log + ((size_t)step * B + v) * 8;
                    r[0] = veh[0]; r[1] = veh[1]; r[2] = veh[2]; r[3] = veh[3]; r[4] = acc_des; r[5] = df_des; r[6] = status[v]; r[7] = iters[v];
                }
            }
            if (final_state) for (int i = 0; i < 8; i++) final_state[8 * v + i] = veh[i];
        }
        return 0;
    }
    std::vector<int> roles(32 * ROLE_STRIDE_F);
    for (int l = 0; l < 32; l++) riccati_roles(l, kc.N, w_sd_of(1, 1), roles.data() + l * ROLE_STRIDE_F, 1);
    kc.roles = roles.data();
    a.pose0 = pose0; a.path_of = path_of;
    a.T = T; a.target_vel = target_vel; a.log = log; a.final_state = final_state; a.B = B;
    std::vector<double> met((size_t)MET_K * B, 0.0 / 0.0);
    const int per_team = smem_doubles_per_team(kc.N, 1, 1);
    std::vector<double> smem_raw((size_t)4 * per_team + 4 * ROLLOUT_PX + 2, 0.0);
    double* smem = smem_raw.data();
    if (((size_t)smem) & 15) smem++;
    for (long b0 = 0; b0 < B; b0 += 4) {
        FWJob j{&kc, &a, b0, smem, per_team, metrics ? met.data() : nullptr, w};
        emu::race_reset();
        for (int q = 0; q < 4; q++) register_benign(smem + (size_t)q * per_team, kc.N, 1);
        emu::run_warp(metrics ? lane_rollout_frenet_w<1> : lane_rollout_frenet_w<0>, &j, 4);
    }
    if (metrics)   // as rollout_metrics_final_kernel
        for (long v = 0; v < B; v++) metrics_finalize(met.data() + v, B, metrics + (size_t)MET_FIELDS * v);
    return 0;
}
