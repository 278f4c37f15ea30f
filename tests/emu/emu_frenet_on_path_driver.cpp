// emu_frenet_on_path_driver.cpp -- TEST ONLY: the reference pass of mpcb200_solve_batch_frenet_on_path (on_path_frenet_ref_kernel:
// frenet_on_path_problem on one warp per problem) on the CPU warp emulator.  It compiles emu_frenet_driver.cpp as it stands (three
// path tables, the host-built fit matrices); the solves of the returned rows are those of emu_driver.cpp and emu_weights_driver.cpp.
#include "emu_frenet_driver.cpp"

struct OPJob { const KCfg* cfg; const FrenetRolloutArgs* a; const double* pose; long b; double* k_out; double* state_out; };
static void lane_frenet_on_path(int, void* p) {
    OPJob* j = (OPJob*)p;
    TeamSolver<1, 1> S(*j->cfg, (smem_t) nullptr);   // (one-warp teams: collectives are shuffles only)
    frenet_on_path_problem(S, *j->a, j->pose, j->b, j->k_out, j->state_out);
}

// B problems: pose [B][4], path_of [B] over the three tables of tb; bit i of unset: table i was never set (n = 0, as
// mpcb200_set_path leaves it).  Out: k_out, state_out [B][4].  Only the fields of FrenetRolloutArgs the kernel fills are set.
extern "C" int emu_frenet_on_path(const KCfg* cfg, const Tables3* tb, int unset, double window, int ey_from_path, long B,
                                  const double* pose, const int* path_of, double* k_out, double* state_out) {
    KCfg kc = *cfg;
    kcfg_finalize(kc);
    std::vector<double> P, cb_store[3];
    const FrenetRolloutArgs full = frenet_args(*tb, window, P, cb_store);
    FrenetRolloutArgs a;
    memset(&a, 0, sizeof(a));
    for (int i = 0; i < 3; i++) a.paths[i] = full.paths[i];
    for (int i = 0; i < 3; i++) if (unset & (1 << i)) memset(&a.paths[i], 0, sizeof(PathTable));
    a.path_of = path_of; a.B = B; a.ey_from_path = ey_from_path;
    a.P1 = full.P1; a.P2 = full.P2; a.n1 = full.n1; a.n2 = full.n2;
    for (long b = 0; b < B; b++) {
        OPJob j{&kc, &a, pose, b, k_out, state_out};
        emu::race_reset();
        emu::run_warp(lane_frenet_on_path, &j, 1);
    }
    return 0;
}
