// tpp_solver.cuh -- the large-batch solve path: ONE THREAD PER PROBLEM, the iterate streamed from HBM.
//
// What it replaces (reference file:line): the same solve(mdl) of scripts/mpc_utils/MKZMPCPathFollower.jl:176 (MODEL 1:
// MKZMPCPathFollowerFrenet.jl:176) as mpc_kernel.cuh, on the same NLP (:65-123), with the same interior-point iteration (Ipopt 3.12 defaults, restated
// formula for formula from TeamSolver::solve) and the same condensed Riccati linear algebra.
//
// Why a second layout.  The warp-per-problem kernel keeps a problem on chip (registers + 18 KB of shared memory), which
// caps an SM at 12 problems, and it spends ~6.5 K warp instructions per interior-point iteration on what is ~17 K scalar
// operations: lanes = stages leaves a third of the lanes idle, lanes = matrix entries turns every 6x6 product into
// shuffles / shared-memory round trips (the kernel is bound by the MIO pipe, profiles/r02_*).  Here a lane owns a whole
// problem: every FP64 instruction does useful work in all 32 lanes, no shuffles, no shared memory; the price is that the
// problem state (~90 doubles per stage) lives in global memory, laid out [warp][stage][field][lane] so that the 32 lanes of a
// warp read and write 256 contiguous bytes per access.  The solve becomes an HBM-streaming
// computation over passes along the horizon:
//     backward pass   stage assembly + Riccati recursion, cost-to-go P (21 + 6 doubles) in registers
//     forward pass    step, fraction-to-the-boundary limits, grad(phi)'d
//     trial pass      model evaluation at the trial point: objective, barrier, constraint violation
//     accept pass     costate recursion (new equality multipliers), iterate / multiplier update, KKT error at the new point
// A normal iteration is exactly one trip through (backward, forward, trial, accept), so lanes that are in different
// iterations of different problems still execute the same instruction stream; extra solves (inertia correction,
// second-order correction) and extra trial points (backtracking) cost the lane that needs them one more trip.
// Lanes are persistent: a lane whose problem ends writes the result and takes the next problem index from a device
// counter, so a slot is always busy while work is left and a problem never changes its slot (coalescing is preserved).
// Measured on the B200 (DESIGN.md 3.7): the layout is HBM-bound (5.5 TB/s at N = 8).  It is at its best when the solves of a batch
// take about the same number of iterations (no tail of long solves once the queue is empty): warm-started batches, closed-loop
// fleets (one control period = plant / waypoints / this solve in place: configs[3] in 0.57 s instead of 1.25 s), and the
// Frenet-frame variant (MODEL 1: 4.8 M instead of 3.2 M solves/s at N = 20, 4.9 TB/s = 75 % of the measured HBM bandwidth).  From the XY model's all-zero start (25 to 200
// iterations) it beats the warp-per-problem kernel at short horizons and large batches (N = 8: 1.5x at 65,536 problems, 2.1x at
// 262,144) and ties with it at N = 20, which is what mpcb200_set_large_batch_path's default rule encodes.
//
// The file is plain scalar C++ behind MPC_DEV, so tests/emu compiles it with g++ and checks it against the oracle
// iterate for iterate on the CPU (tests/test_tpp_emu.py).
#pragma once
#include "mpc_kernel.cuh"

#ifdef MPC_HOST_EMU
#define MPC_UNROLL
#else
#define MPC_UNROLL _Pragma("unroll")
#endif

namespace mpcb200 {

// ---- per-stage fields of a slot's state
enum {
    TF_SX = 0, TF_SY, TF_SP, TF_SV, TF_UA, TF_UD,          // primal iterate
    TF_YX, TF_YY, TF_YP, TF_YV,                            // multipliers of the equality rows that define s_k
    TF_RS0, TF_RS1, TF_RY0, TF_RY1,                        // rate row ending at u_k: slack, multiplier ([0] steering, [1] acceleration)
    TF_ZVL, TF_ZVU, TF_ZAL, TF_ZAU, TF_ZDL, TF_ZDU, TF_RVL0, TF_RVL1, TF_RVU0, TF_RVU1,   // bound multipliers
    TF_XR, TF_YR, TF_PR,                                   // reference sample
    TF_DX, TF_DY, TF_DP, TF_DV, TF_DA, TF_DD, TF_DRS0, TF_DRS1,   // step (primal, rate-row slacks)
    TF_K,                                                  // 14 gains: K[0][0..6], K[1][0..6]
    TF_GX = TF_K + 14, TF_GY, TF_GP, TF_GV, TF_GA, TF_GD,  // condensed gradient of the last assembled system
    TF_HPP, TF_HPV, TF_HVV, TF_HPD, TF_HVD,                // ... its condensed Hessian entries that are not constants
    TF_SRW0, TF_SRW1, TF_BR0, TF_BR1,                      // ... (Sigma_s + delta_w) and barrier gradient of the rate rows
    TF_C,                                                  // 6: second-order-correction right-hand side (rd[4], dr[2])
    TF_EV = TF_C + 6                                       // 2 x TEV_N: model evaluation at the current / the trial point
};
enum { TEV_CS = 0, TEV_SN, TEV_CB, TEV_SB, TEV_B1, TEV_B2, TEV_RD, TEV_DR = TEV_RD + 4, TEV_Q = TEV_DR + 2, TEV_K };
// MODEL 1 (Frenet-frame variant, MKZMPCPathFollowerFrenet.jl): the evaluation also holds q = 1 / (1 - e_y K(s)) and K(s), and the
// condensed Hessian has nine more entries that are constants or zeros in the XY model
enum { TFH_SS = 0, TFH_EE, TFH_SE, TFH_SP, TFH_SV, TFH_SD, TFH_EP, TFH_EV, TFH_ED, TFH_N };
MPC_HD constexpr int tev_n(int model) { return model ? 14 : 12; }
MPC_HD constexpr int tf_fh(int model) { return TF_EV + 2 * tev_n(model); }               // first of the TFH_* fields (MODEL 1)
MPC_HD constexpr int tf_nfield(int model) { return tf_fh(model) + (model ? TFH_N : 0); }
#define TPP_NFILT 32   // filter entries per problem (as many as the one-warp kernel holds)

// Layout: [warp][stage][field][lane].  A warp owns one contiguous region; the 32 lanes of an access are 256 contiguous
// bytes, a stage's fields sit 256 bytes apart (so every field of the current and the neighbouring stages is an immediate
// offset from one per-stage pointer: no address arithmetic per access), and a warp walks its region linearly.
template <int MODEL>
struct TppMemT {
    static constexpr int NF = tf_nfield(MODEL);
    double* wb;     // this lane's element of field 0, stage 0 of its warp's region
    double* fb;     // ... of filter entry 0
    MPC_DEV TppMemT(double* st, double* filt, int N, long slot)
        : wb(st + (slot >> 5) * ((long)(N + 1) * NF * 32) + (slot & 31)), fb(filt + (slot >> 5) * (2L * TPP_NFILT * 32) + (slot & 31)) {}
    MPC_DEV double ld(int f, int k) const { return (wb + (long)k * (NF * 32))[f * 32]; }
    MPC_DEV void sto(int f, int k, double v) const { (wb + (long)k * (NF * 32))[f * 32] = v; }
    // L2 prefetch of fields [f0, f0 + nf) of stage k for the whole warp (one bulk instruction from one active lane).  Off by
    // default: it never paid (the stage bodies issue all their loads up front, which covers the latency), and once the kernel was
    // HBM-bound the fields a coarse range fetches without need cost 3-5 % (profiles/r02_logs/r02_tpp_noprefetch.log);
    // -DMPC_TPP_PREFETCH=<mask of passes: 1 trial, 2 backward, 4 forward, 8 accept> brings it back.  The backward pass's ranges are
    // exactly what it loads, and prefetching only those changes nothing either (13.73 vs 13.76 ms, r02_tpp_prefetch_per_pass.log)
    template <int PASS>
    MPC_DEV void prefetch(int k, int f0, int nf) const {
#if !defined(MPC_HOST_EMU) && defined(MPC_TPP_PREFETCH)
        if (!((MPC_TPP_PREFETCH) & PASS)) return;
        const unsigned am = __activemask();
        const int lane = threadIdx.x & 31;
        if (lane == __ffs(am) - 1)
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(wb - lane + ((long)k * NF + f0) * 32), "r"(nf * 256) : "memory");
#else
        (void)k; (void)f0; (void)nf;
#endif
    }
    MPC_DEV double fld(int e) const { return fb[e * 32]; }
    MPC_DEV void fst(int e, double v) const { fb[e * 32] = v; }
};
typedef TppMemT<0> TppMem;
// slots are rounded up to whole warps
MPC_HD size_t tpp_state_doubles(int N, long S, int model = 0) { return (size_t)tf_nfield(model) * (size_t)(N + 1) * (size_t)((S + 31) / 32 * 32); }
MPC_HD size_t tpp_filter_doubles(long S) { return (size_t)2 * TPP_NFILT * (size_t)((S + 31) / 32 * 32); }

struct TrueT { static constexpr bool value = true; };
struct FalseT { static constexpr bool value = false; };
MPC_DEV double nanmax(double v, double t) { return (t > v || t != t) ? t : v; }   // NaN wins, like warp_max
MPC_DEV constexpr int sidx(int i, int j) { return (i <= j) ? (i * 6 - i * (i - 1) / 2 + (j - i)) : (j * 6 - j * (j - 1) / 2 + (i - j)); }

// PW: the cost weights are the problem's own row `wr` (BatchPtrs::w; KCfg::w when it is null), read from global memory where they are
// used (64 bytes per problem against the ~43 KB of slot state a trip streams); PW = 0 reads the kernel parameter KCfg::w
template <int MODEL = 0, int PW = 0>
struct TppSolverT {
    static constexpr int TEVN = tev_n(MODEL), TF_FH = tf_fh(MODEL);
    const KCfg& c;
    const TppMemT<MODEL> m;
    const int N;
    const double* wr;   // PW: this problem's weight row (row_weight layout of its model) or null
    double cst[7];   // state[4], u_prev (df, acc), v_des
    double kp[4];    // MODEL 1: the problem's curvature polynomial K(s), highest degree first
    // ---- interior-point driver state (TeamSolver::solve's locals)
    double sigma, mu, tau, dw, dw_last, theta_max, theta_min, phi, gBd, alpha, alpha_max, Rft, a_soc, th_soc_old;
    double cur_theta, cur_f, cur_lb, ev_f, ev_lb, ev_theta, ev_alpha;
    double p2_amax, p2_az, p2_gBd;                        // by-products of the forward pass
    double e_di, e_cv, e_pzabs, e_pzmax, e_pzmin, e_sumy, e_sumz, e_xm, e_ym;   // KKT error pieces at the current point
    int phase, op, acc_mode, req, nfilt, accept_count, iter, nsteps, soc_cnt, n_resto, evcur, ret;
    bool soc_first, resto_check, cur_acceptable, had_acceptable, tiny_last, tiny, p2_tiny, solve_ok, feasible, ls_system;
    enum { PH_INIT = 0, PH_EVAL0, PH_LS, PH_BEGIN, PH_PD, PH_RESOLVE, PH_TRIAL, PH_SOC, PH_RESTO };
    enum { RUNNING = -100 };

    MPC_DEV TppSolverT(const KCfg& cfg, const TppMemT<MODEL>& mem) : c(cfg), m(mem), N(cfg.N), wr(nullptr) {}

    MPC_DEV bool isU(int k) const { return k < N; }
    MPC_DEV bool isR(int k) const { return (k == 0 || k >= 2) && k < N; }
    MPC_DEV double wt(int i) const { return (PW && wr) ? row_weight(wr, 0, i, MODEL) : c.w[i]; }   // cost weight i (update_cost order)
    MPC_DEV double wx(int k) const { return (k >= 1) ? wt(0) : 0.0; }
    MPC_DEV double wy(int k) const { return (k >= 1) ? wt(1) : 0.0; }
    MPC_DEV double wp(int k) const { return (k >= 1) ? wt(2) : 0.0; }
    MPC_DEV double wv(int k) const { return (k >= 1 && k <= N - 1) ? wt(3) : 0.0; }
    MPC_DEV double rHi(int k, int i) const { return (k == 0) ? c.rHiFirst[i] : c.rHiLater[i]; }
    MPC_DEV int evb(int which) const { return TF_EV + TEVN * which; }
    // reference sample of stage k; MODEL 1: the cost is on e_y, e_psi themselves (reference 0): nothing to read
    MPC_DEV double ref(int f, int k) const { return MODEL ? 0.0 : m.ld(f, k); }

    // MODEL 1 (MKZMPCPathFollowerFrenet.jl:111-120): curvature K(s) of the problem's cubic and its derivatives; the stage
    // Jacobian of  ds/dt = g = v cos(e_psi + beta) / (1 - e_y K(s)),  d e_psi/dt = v sin(beta) / L_b - g K  at a stage that owns an
    // input (TeamSolver::frenet_jac, same expressions)
    struct Curv { double K, K1, K2; };
    MPC_DEV Curv curvature(double s) const {
        Curv r;
        r.K = ((kp[0] * s + kp[1]) * s + kp[2]) * s + kp[3];
        r.K1 = (3.0 * kp[0] * s + 2.0 * kp[1]) * s + kp[2];
        r.K2 = 6.0 * kp[0] * s + 2.0 * kp[1];
        return r;
    }
    struct FJac { double a00, a01, a02, a03, a12, a13, a20, a21, a22, a23, b0, b1, b2, G0, G1, G2, G3, G4, g, K1, K2; };
    MPC_DEV FJac frenet_jac(double cs, double sn, double cb, double sb, double b1e, double q, double K, double s, double ey, double v) const {
        FJac J;
        const Curv cu = curvature(s);
        const double dt = c.dt;
        const double q2 = q * q;
        const double qs = ey * cu.K1 * q2, qe = K * q2;
        J.K1 = cu.K1; J.K2 = cu.K2;
        J.g = v * cs * q;
        J.G0 = v * cs * qs; J.G1 = v * cs * qe; J.G2 = -v * sn * q; J.G3 = cs * q; J.G4 = -v * sn * b1e * q;
        J.a00 = 1.0 + dt * J.G0; J.a01 = dt * J.G1; J.a02 = dt * J.G2; J.a03 = dt * J.G3; J.b0 = dt * J.G4;
        J.a12 = dt * v * cs; J.a13 = dt * sn; J.b1 = dt * v * cs * b1e;
        J.a20 = -dt * (J.G0 * K + J.g * cu.K1); J.a21 = -dt * J.G1 * K; J.a22 = 1.0 - dt * J.G2 * K;
        J.a23 = dt * (sb / c.Lb - J.G3 * K); J.b2 = dt * (v * cb * b1e / c.Lb - J.G4 * K);
        return J;
    }

    // reciprocals of the ten bound slacks of stage k from one division (TeamSolver::recips)
    MPC_DEV void recips(int k, bool u, bool r, double sv, double ua, double ud, double rs0, double rs1, Recips& q) const {
        const double vl = sv - c.vLo, vu = c.vHi - sv;
        const double al = u ? ua - c.aLo : 1.0, au = u ? c.aHi - ua : 1.0;
        const double dl = u ? ud - c.dLo : 1.0, du = u ? c.dHi - ud : 1.0;
        const double h0 = rHi(k, 0), h1 = rHi(k, 1);
        const double r0l = r ? rs0 + h0 : 1.0, r0u = r ? h0 - rs0 : 1.0;
        const double r1l = r ? rs1 + h1 : 1.0, r1u = r ? h1 - rs1 : 1.0;
        const double pv = vl * vu, pa_ = al * au, pd_ = dl * du, p0 = r0l * r0u, p1 = r1l * r1u;
        const double pva = pv * pa_, p01 = p0 * p1, pvad = pva * pd_;
        const double iall = 1.0 / (pvad * p01);
        const double i01 = iall * pvad, ivad = iall * p01;
        const double ip0 = i01 * p1, ip1 = i01 * p0;
        const double ipd = ivad * pva, iva = ivad * pd_;
        const double ipv = iva * pa_, ipa = iva * pv;
        q.vL = vu * ipv; q.vU = vl * ipv; q.aL = au * ipa; q.aU = al * ipa; q.dL = du * ipd; q.dU = dl * ipd;
        q.r0L = r0u * ip0; q.r0U = r0l * ip0; q.r1L = r1u * ip1; q.r1U = r1l * ip1;
    }

    // ------------------------------------------------------------------
    // problem set-up: inputs into the slot, driver state reset, first driver step (interior start)
    // ------------------------------------------------------------------
    MPC_DEV void begin(const BatchPtrs& io, long b, double v_des0 = 0.0) {
        const long nr = 3L * (N + 1), nt = 6L * N + 4;
        if (PW) wr = io.w ? io.w + (MODEL ? 7 : 8) * b : nullptr;
        for (int i = 0; i < 4; i++) cst[i] = io.state[4 * b + i];
        cst[4] = io.u_prev[2 * b]; cst[5] = io.u_prev[2 * b + 1];
        cst[6] = io.v_des ? io.v_des[b] : v_des0;
        // MODEL 1: io.ref = [B][4] curvature polynomial; the cost is on e_y, e_psi themselves (reference 0)
        const double* rf = MODEL ? io.ref + 4 * b : io.ref + nr * b;
        if (MODEL) for (int i = 0; i < 4; i++) kp[i] = rf[i];
        const double* w = io.warm ? io.warm + nt * b : nullptr;
        for (int k = 0; k <= N; k++) {
            m.sto(TF_XR, k, MODEL ? 0.0 : rf[k]); m.sto(TF_YR, k, MODEL ? 0.0 : rf[(N + 1) + k]); m.sto(TF_PR, k, MODEL ? 0.0 : rf[2 * (N + 1) + k]);
            m.sto(TF_SX, k, w ? w[k] : 0.0); m.sto(TF_SY, k, w ? w[(N + 1) + k] : 0.0);
            m.sto(TF_SV, k, w ? w[2 * (N + 1) + k] : 0.0); m.sto(TF_SP, k, w ? w[3 * (N + 1) + k] : 0.0);
            m.sto(TF_UD, k, (w && k < N) ? w[4 * (N + 1) + k] : 0.0); m.sto(TF_UA, k, (w && k < N) ? w[4 * (N + 1) + N + k] : 0.0);
        }
        if (!w && c.start_mode == 1) {   // MPCB200_START_ROLLOUT: previous command held over the horizon, rolled out
            for (int k = 0; k < N; k++) { m.sto(TF_UA, k, cst[5]); m.sto(TF_UD, k, cst[4]); }
            rollout_restore();
        }
        prologue();
    }

    // A problem whose reference samples are already in the slot (written by the waypoint kernel of a closed-loop step) and
    // whose start point is either `warm0` ([6N+4], the layout of BatchPtrs::warm) or whatever the slot holds -- the
    // previous solution of the same vehicle: the control loop's warm start without moving a byte.  (PW: the caller sets wr.)
    MPC_DEV void begin_in_place(const double c7[7], const double* warm0) {
        for (int i = 0; i < 7; i++) cst[i] = c7[i];
        if (warm0) {
            for (int k = 0; k <= N; k++) {
                m.sto(TF_SX, k, warm0[k]); m.sto(TF_SY, k, warm0[(N + 1) + k]);
                m.sto(TF_SV, k, warm0[2 * (N + 1) + k]); m.sto(TF_SP, k, warm0[3 * (N + 1) + k]);
                m.sto(TF_UD, k, (k < N) ? warm0[4 * (N + 1) + k] : 0.0); m.sto(TF_UA, k, (k < N) ? warm0[4 * (N + 1) + N + k] : 0.0);
            }
        }
        prologue();
    }

    // TeamSolver::solve's prologue: feasibility of the NLP, objective scaling from the gradient at the start point, driver reset
    MPC_DEV void prologue() {
        feasible = nlp_feasible();
        ret = feasible ? RUNNING : 2;
        sigma = 1.0;
        {
            double gm = 0.0, pa = 0.0, pd = 0.0;
            double ua = m.ld(TF_UA, 0), ud = m.ld(TF_UD, 0);
            for (int k = 0; k <= N; k++) {
                const double na = (k + 1 < N) ? m.ld(TF_UA, k + 1) : 0.0, nd = (k + 1 < N) ? m.ld(TF_UD, k + 1) : 0.0;
                const Grad g = objective_gradient(k, isU(k), m.ld(TF_SX, k), m.ld(TF_SY, k), m.ld(TF_SP, k), m.ld(TF_SV, k), ua, ud, pa, pd, na, nd);
                double t = dmax_(dmax_(fabs(g.x), fabs(g.y)), dmax_(fabs(g.p), fabs(g.v)));
                t = dmax_(t, dmax_(fabs(g.a), fabs(g.d)));
                gm = nanmax(gm, t);
                pa = ua; pd = ud; ua = na; ud = nd;
            }
            sigma = (gm > K_SCALE_MAX_GRAD) ? dmax_(K_SCALE_MAX_GRAD / gm, 1e-8) : 1.0;
        }
        phase = PH_INIT; op = OP_INIT; acc_mode = 0;
        soc_first = resto_check = cur_acceptable = had_acceptable = false;
        n_resto = 0; req = 0; ev_alpha = 0.0; evcur = 0; ls_system = false;
        mu = K_MU_INIT; tau = dmax_(K_TAU_MIN, 1.0 - K_MU_INIT);
        dw = 0.0; dw_last = 0.0; theta_max = -1.0; theta_min = -1.0;
        nfilt = 0; accept_count = 0; iter = 0;
        tiny_last = tiny = solve_ok = false;
        cur_theta = cur_f = cur_lb = 0.0; phi = gBd = 0.0; alpha = alpha_max = 1.0; Rft = 0.0; a_soc = 0.0; th_soc_old = 0.0;
        nsteps = soc_cnt = 0;
        for (int k = 0; k <= N; k++) {   // multipliers and slacks of a fresh solve
            m.sto(TF_YX, k, 0.0); m.sto(TF_YY, k, 0.0); m.sto(TF_YP, k, 0.0); m.sto(TF_YV, k, 0.0);
            m.sto(TF_RS0, k, 0.0); m.sto(TF_RS1, k, 0.0); m.sto(TF_RY0, k, 0.0); m.sto(TF_RY1, k, 0.0);
        }
    }

    MPC_DEV bool nlp_feasible() const {
        const double e = 1e-8;
        const double lim_d = c.sdmax * c.dtc, lim_a = c.admax * c.dtc;
        const double v0 = cst[3], up0 = cst[4], up1 = cst[5];
        if (v0 < c.vmin - e * dmax_(1.0, fabs(c.vmin))) return false;
        if (v0 > c.vmax + e * dmax_(1.0, fabs(c.vmax))) return false;
        if (up0 - lim_d > c.smax + 2 * e || up0 + lim_d < -c.smax - 2 * e) return false;
        if (up1 - lim_a > c.amax + 2 * e || up1 + lim_a < -c.amax - 2 * e) return false;
        return true;
    }

    // scaled objective gradient of stage k (MKZMPCPathFollower.jl:97-103; rate terms counted at both inputs they couple)
    struct Grad { double x, y, p, v, a, d; };
    MPC_DEV Grad objective_gradient(int k, bool u, double sx, double sy, double sp, double sv, double ua, double ud, double pa, double pd, double na, double nd) const {
        Grad g;
        const double s2 = 2.0 * sigma;
        g.x = s2 * wx(k) * (sx - ref(TF_XR, k));
        g.y = s2 * wy(k) * (sy - ref(TF_YR, k));
        g.p = s2 * wp(k) * (sp - ref(TF_PR, k));
        g.v = s2 * wv(k) * (sv - cst[6]);
        g.a = 0.0; g.d = 0.0;
        if (u) {
            g.a = s2 * wt(6) * ua;
            g.d = s2 * wt(7) * ud;
            if (k >= 1) { g.a += s2 * wt(4) * (ua - pa); g.d += s2 * wt(5) * (ud - pd); }
            if (k + 1 < N) { g.a -= s2 * wt(4) * (na - ua); g.d -= s2 * wt(5) * (nd - ud); }
        }
        return g;
    }

    // ------------------------------------------------------------------
    // interior start (DefaultIterateInitializer): push into the interior, slacks = d(x) pushed, z = 1, zero step
    // ------------------------------------------------------------------
    MPC_DEV void init_pass() {
        double pa = 0.0, pd = 0.0;
        for (int k = 0; k <= N; k++) {
            double sv = m.ld(TF_SV, k);
            push_interior(sv, c.vLo, c.vHi);
            m.sto(TF_SV, k, sv);
            double ua = 0.0, ud = 0.0;
            if (isU(k)) {
                ua = m.ld(TF_UA, k); ud = m.ld(TF_UD, k);
                push_interior(ua, c.aLo, c.aHi); push_interior(ud, c.dLo, c.dHi);
                m.sto(TF_UA, k, ua); m.sto(TF_UD, k, ud);
            }
            const bool r = isR(k);
            if (r) {
                const double h0 = rHi(k, 0), h1 = rHi(k, 1);
                double rs0 = ud - ((k == 0) ? cst[4] : pd), rs1 = ua - ((k == 0) ? cst[5] : pa);
                push_interior(rs0, -h0, h0); push_interior(rs1, -h1, h1);
                m.sto(TF_RS0, k, rs0); m.sto(TF_RS1, k, rs1);
            }
            const double zu = isU(k) ? 1.0 : 0.0, zr = r ? 1.0 : 0.0;
            m.sto(TF_ZVL, k, 1.0); m.sto(TF_ZVU, k, 1.0);
            m.sto(TF_ZAL, k, zu); m.sto(TF_ZAU, k, zu); m.sto(TF_ZDL, k, zu); m.sto(TF_ZDU, k, zu);
            m.sto(TF_RVL0, k, zr); m.sto(TF_RVL1, k, zr); m.sto(TF_RVU0, k, zr); m.sto(TF_RVU1, k, zr);
            for (int f = TF_DX; f <= TF_DRS1; f++) m.sto(f, k, 0.0);
            pa = ua; pd = ud;
        }
    }

    // ------------------------------------------------------------------
    // The four passes along the horizon.  Every stage body is written as  loads -> arithmetic -> stores : the loads of
    // a body are independent of everything computed in it, and a load that follows a store to the same array cannot be
    // moved above it by the compiler, so the source order is what lets all of a body's loads be in flight together
    // (one exposed memory latency per stage and pass instead of one per group of fields).
    // ------------------------------------------------------------------

    // trial pass: model evaluation at  L + a D  into the trial buffer; objective, log-barrier, violation
    MPC_DEV void eval_pass(double a) {
        const int eb = evb(evcur ^ 1);
        double f = 0.0, lb = 0.0, th = 0.0;
        double sx = m.ld(TF_SX, 0) + a * m.ld(TF_DX, 0), sy = m.ld(TF_SY, 0) + a * m.ld(TF_DY, 0);
        double sp = m.ld(TF_SP, 0) + a * m.ld(TF_DP, 0), sv = m.ld(TF_SV, 0) + a * m.ld(TF_DV, 0);
        double pa = cst[5], pd = cst[4];   // previous input as the rate rows see it
        const double i0 = cst[0] - sx, i1 = cst[1] - sy, i2 = cst[2] - sp, i3 = cst[3] - sv;
        th = fabs(i0) + fabs(i1) + fabs(i2) + fabs(i3);
        // the body is instantiated twice: for the stages that own an input (the loop) and for the terminal stage, so
        // that everything that depends on "has an input" folds at compile time
        auto body = [&](const int k, auto UT) {
            constexpr bool u = decltype(UT)::value;
            const bool r = u && isR(k);
            if (k + 2 <= N) m.template prefetch<1>(k + 2, 0, TF_K);
            // ---- loads
            const double xr = ref(TF_XR, k), yr = ref(TF_YR, k), pr = ref(TF_PR, k);
            double ua = 0.0, ud = 0.0, s0 = 0.0, s1 = 0.0;
            double nx = 0.0, ny = 0.0, np = 0.0, nv = 0.0;
            if (u) {
                const double ua0 = m.ld(TF_UA, k), ud0 = m.ld(TF_UD, k), da = m.ld(TF_DA, k), dd = m.ld(TF_DD, k);
                const double x1 = m.ld(TF_SX, k + 1), y1 = m.ld(TF_SY, k + 1), p1 = m.ld(TF_SP, k + 1), v1 = m.ld(TF_SV, k + 1);
                const double dx1 = m.ld(TF_DX, k + 1), dy1 = m.ld(TF_DY, k + 1), dp1 = m.ld(TF_DP, k + 1), dv1 = m.ld(TF_DV, k + 1);
                const double rs0 = m.ld(TF_RS0, k), rs1 = m.ld(TF_RS1, k), drs0 = m.ld(TF_DRS0, k), drs1 = m.ld(TF_DRS1, k);
                ua = ua0 + a * da; ud = ud0 + a * dd;
                nx = x1 + a * dx1; ny = y1 + a * dy1; np = p1 + a * dp1; nv = v1 + a * dv1;
                s0 = rs0 + a * drs0; s1 = rs1 + a * drs1;
            }
            // ---- arithmetic
            double rd0 = 0.0, rd1 = 0.0, rd2 = 0.0, rd3 = 0.0, dr0 = 0.0, dr1 = 0.0;
            double cs = 0.0, sn = 0.0, cb = 0.0, sb = 0.0, b1 = 0.0, b2 = 0.0, qv = 0.0, Kv = 0.0;
            if (u) {
                // beta = atan(r tan df) in closed form, valid for |df| < pi/2 (bounds keep |df| <= 0.5)
                const double rr = c.rfrac;
                double sd, cd, sps, cps;
                mpc_sincos(ud, &sd, &cd);
                mpc_sincos(sp, &sps, &cps);
                const double Dn = cd * cd + rr * rr * sd * sd;
                const double iD = 1.0 / Dn;
                const double inv = sqrt(iD);
                cb = cd * inv; sb = rr * sd * inv;
                cs = cps * cb - sps * sb; sn = sps * cb + cps * sb;
                b1 = rr * iD; b2 = rr * (1.0 - rr * rr) * (2.0 * sd * cd) * (iD * iD);
                double fx = sx + c.dt * (sv * cs), fp = sp + c.dtLb * (sv * sb);
                const double fy = sy + c.dt * (sv * sn), fv = sv + c.dt * ua;
                if (MODEL) {   // MKZMPCPathFollowerFrenet.jl:111-120: ds/dt = v cos(e_psi + beta) / (1 - e_y K(s))
                    Kv = curvature(sx).K;
                    qv = 1.0 / (1.0 - sy * Kv);
                    const double g = sv * cs * qv;
                    fx = sx + c.dt * g;
                    fp = sp + c.dt * (sv * sb / c.Lb - g * Kv);
                }
                rd0 = fx - nx; rd1 = fy - ny; rd2 = fp - np; rd3 = fv - nv;
            }
            if (r) { dr0 = (ud - pd) - s0; dr1 = (ua - pa) - s1; }
            // objective (MKZMPCPathFollower.jl:97-103): stage terms + rate terms counted at the later input
            {
                const double ex = sx - xr, ey = sy - yr, ep = sp - pr, evv = sv - cst[6];
                double fk = wx(k) * ex * ex + wy(k) * ey * ey + wp(k) * ep * ep + wv(k) * evv * evv;
                if (u) {
                    fk += wt(6) * ua * ua + wt(7) * ud * ud;
                    if (k >= 1) { const double da = ua - pa, dd = ud - pd; fk += wt(4) * da * da + wt(5) * dd * dd; }
                }
                f += fk;
            }
            double p = (sv - c.vLo) * (c.vHi - sv);
            if (u) p *= (ua - c.aLo) * (c.aHi - ua) * (ud - c.dLo) * (c.dHi - ud);
            if (r) { const double h0 = rHi(k, 0), h1 = rHi(k, 1); p *= (s0 + h0) * (h0 - s0) * (s1 + h1) * (h1 - s1); }
            lb += log(p);
            th += fabs(rd0) + fabs(rd1) + fabs(rd2) + fabs(rd3) + fabs(dr0) + fabs(dr1);
            // ---- stores
            if (u) {
                m.sto(eb + TEV_CS, k, cs); m.sto(eb + TEV_SN, k, sn); m.sto(eb + TEV_CB, k, cb); m.sto(eb + TEV_SB, k, sb);
                m.sto(eb + TEV_B1, k, b1); m.sto(eb + TEV_B2, k, b2);
                m.sto(eb + TEV_RD + 0, k, rd0); m.sto(eb + TEV_RD + 1, k, rd1); m.sto(eb + TEV_RD + 2, k, rd2); m.sto(eb + TEV_RD + 3, k, rd3);
                m.sto(eb + TEV_DR, k, dr0); m.sto(eb + TEV_DR + 1, k, dr1);
                if (MODEL) { m.sto(eb + TEV_Q, k, qv); m.sto(eb + TEV_K, k, Kv); }
            } else {   // slot N of the evaluation holds the initial-condition residual
                m.sto(eb + TEV_RD + 0, k, i0); m.sto(eb + TEV_RD + 1, k, i1); m.sto(eb + TEV_RD + 2, k, i2); m.sto(eb + TEV_RD + 3, k, i3);
            }
            sx = nx; sy = ny; sp = np; sv = nv; pa = ua; pd = ud;
        };
        MPC_NOUNROLL for (int k = 0; k < N; k++) body(k, TrueT{});
        body(N, FalseT{});
        ev_f = f; ev_lb = lb; ev_theta = th;
    }

    // ------------------------------------------------------------------
    // backward pass: stage assembly (TeamSolver::assemble) fused with the Riccati recursion
    // (TeamSolver::riccati_backward).  Returns false if some stage's reduced input Hessian is not positive
    // definite (= wrong inertia of the KKT matrix).
    //   rq 0: least-squares multiplier system; rq 1, 2: primal-dual system; rq 3: ... with the second-order-correction
    //   right-hand side
    // ------------------------------------------------------------------
    MPC_DEV bool backward_pass(int rq) {
        const int ec = evb(evcur);
        const bool ls = (rq == 0), soc = (rq == 3);
        const int rb = soc ? TF_C : ec + TEV_RD, db = soc ? TF_C + 4 : ec + TEV_DR;   // where the right-hand-side residuals are
        const double s2 = 2.0 * sigma;
        double P[21], pv[6];
        MPC_UNROLL for (int i = 0; i < 21; i++) P[i] = 0.0;
        MPC_UNROLL for (int i = 0; i < 6; i++) pv[i] = 0.0;
        double y1x = 0.0, y1y = 0.0, y1p = 0.0;   // multipliers of the rows leaving stage k (held by stage k + 1)
        double wn0 = 0.0, wn1 = 0.0;              // rate-row term of stage k + 1
        double na = 0.0, nd = 0.0;                // inputs of stage k + 1
        double ua = 0.0, ud = 0.0;                // inputs of stage k (loaded one stage ahead)
        auto body = [&](const int k, auto UT) -> bool {
            constexpr bool u = decltype(UT)::value;
            const bool r = u && isR(k);
            if (k >= 1) { m.template prefetch<2>(k - 1, 0, TF_DX); m.template prefetch<2>(k - 1, soc ? TF_C : ec, soc ? 6 : TEVN); }
            // ---- loads
            const int kp = (k >= 1) ? k - 1 : 0;
            const double sx = m.ld(TF_SX, k), sy = m.ld(TF_SY, k), sp = m.ld(TF_SP, k), sv = m.ld(TF_SV, k);
            const double pa = m.ld(TF_UA, kp), pd = m.ld(TF_UD, kp);   // (not used at k = 0)
            const double xr = ref(TF_XR, k), yr = ref(TF_YR, k), pr = ref(TF_PR, k);
            const double yxk = m.ld(TF_YX, k), yyk = m.ld(TF_YY, k), ypk = m.ld(TF_YP, k);
            const double zvL = m.ld(TF_ZVL, k), zvU = m.ld(TF_ZVU, k);
            double zaL = 0.0, zaU = 0.0, zdL = 0.0, zdU = 0.0, rvL0 = 0.0, rvL1 = 0.0, rvU0 = 0.0, rvU1 = 0.0, rs0 = 0.0, rs1 = 0.0;
            double cs = 0.0, sn = 0.0, cb = 0.0, sb = 0.0, b1 = 0.0, b2 = 0.0, eq = 0.0, eK = 0.0;
            double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0, rdr0 = 0.0, rdr1 = 0.0;
            if (u) {
                zaL = m.ld(TF_ZAL, k); zaU = m.ld(TF_ZAU, k); zdL = m.ld(TF_ZDL, k); zdU = m.ld(TF_ZDU, k);
                rvL0 = m.ld(TF_RVL0, k); rvL1 = m.ld(TF_RVL1, k); rvU0 = m.ld(TF_RVU0, k); rvU1 = m.ld(TF_RVU1, k);
                rs0 = m.ld(TF_RS0, k); rs1 = m.ld(TF_RS1, k);
                cs = m.ld(ec + TEV_CS, k); sn = m.ld(ec + TEV_SN, k); cb = m.ld(ec + TEV_CB, k); sb = m.ld(ec + TEV_SB, k);
                b1 = m.ld(ec + TEV_B1, k); b2 = m.ld(ec + TEV_B2, k);
                if (MODEL) { eq = m.ld(ec + TEV_Q, k); eK = m.ld(ec + TEV_K, k); }
                r0 = m.ld(rb + 0, k); r1 = m.ld(rb + 1, k); r2 = m.ld(rb + 2, k); r3 = m.ld(rb + 3, k);
                rdr0 = m.ld(db, k); rdr1 = m.ld(db + 1, k);
                if (ls) { r0 = r1 = r2 = r3 = 0.0; }
                if (ls || !r) { rdr0 = rdr1 = 0.0; }
                if (!r) { rvL0 = rvL1 = rvU0 = rvU1 = 0.0; rs0 = rs1 = 0.0; }
            }
            // ---- arithmetic
            if (!u) { ua = 0.0; ud = 0.0; }
            FJac J;
            if (MODEL && u) J = frenet_jac(cs, sn, cb, sb, b1, eq, eK, sx, sy, sv);
            Grad g;
            {
                g.x = s2 * wx(k) * (sx - xr); g.y = s2 * wy(k) * (sy - yr); g.p = s2 * wp(k) * (sp - pr); g.v = s2 * wv(k) * (sv - cst[6]);
                g.a = 0.0; g.d = 0.0;
                if (u) {
                    g.a = s2 * wt(6) * ua;
                    g.d = s2 * wt(7) * ud;
                    if (k >= 1) { g.a += s2 * wt(4) * (ua - pa); g.d += s2 * wt(5) * (ud - pd); }
                    if (k + 1 < N) { g.a -= s2 * wt(4) * (na - ua); g.d -= s2 * wt(5) * (nd - ud); }
                }
            }
            double Hxx, Hyy, Hpp, Hpv = 0.0, Hvv, Hpd = 0.0, Hvd = 0.0, Haa, Hdd, Ca = 0.0, Cd = 0.0;
            double hss = 0.0, hee = 0.0, Hse = 0.0, Hsp = 0.0, Hsv = 0.0, Hsd = 0.0, Hep = 0.0, Hev = 0.0, Hed = 0.0;   // MODEL 1 only
            double gsv, gua = 0.0, gud = 0.0;
            double SrW0 = 0.0, SrW1 = 0.0, br0 = 0.0, br1 = 0.0, wrow0 = 0.0, wrow1 = 0.0;
            if (ls) {
                if (r) { SrW0 = SrW1 = 1.0; br0 = -(rvL0 - rvU0); br1 = -(rvL1 - rvU1); wrow0 = br0; wrow1 = br1; }
                Hxx = Hyy = Hpp = Hvv = 1.0;
                Ca = (u && r) ? 1.0 : 0.0; Cd = Ca;
                Haa = 1.0 + Ca; Hdd = 1.0 + Cd;
                gsv = g.v + (-zvL + zvU);
                if (u) { gua = g.a - zaL + zaU; gud = g.d - zdL + zdU; }
            } else {
                double hpp = 0.0, hdd = 0.0;
                if (MODEL && u) {
                    // Lagrangian Hessian of the Frenet stage map over (s, e_y, e_psi, v, df): with g = v C q, rows s and e_psi contribute
                    //   -dt [ (y_s - y_p K) hess g - y_p K' (e_s grad g' + grad g e_s') - y_p g K'' e_s e_s' ]   (TeamSolver::assemble)
                    const double v = sv, dt = c.dt, q = eq, K = eK, Cc = cs, Sc = sn, ey = sy;
                    const double q2 = q * q, q3 = q2 * q, K1 = J.K1, K2 = J.K2;
                    const double qs = ey * K1 * q2, qe = K * q2;
                    const double qss = ey * K2 * q2 + 2.0 * ey * ey * K1 * K1 * q3, qse = K1 * q2 + 2.0 * ey * K * K1 * q3, qee = 2.0 * K * K * q3;
                    const double mm = y1x - y1p * K, nn = y1p * K1;
                    hss = -dt * (mm * (v * Cc * qss) - 2.0 * nn * J.G0 - y1p * J.g * K2);
                    Hse = -dt * (mm * (v * Cc * qse) - nn * J.G1);
                    Hsp = -dt * (mm * (-v * Sc * qs) - nn * J.G2);
                    Hsv = -dt * (mm * (Cc * qs) - nn * J.G3);
                    Hsd = -dt * (mm * (-v * Sc * b1 * qs) - nn * J.G4);
                    hee = -dt * mm * (v * Cc * qee);
                    Hep = dt * mm * (v * Sc * qe); Hev = -dt * mm * (Cc * qe); Hed = dt * mm * (v * Sc * b1 * qe);
                    hpp = dt * mm * (v * Cc * q) + y1y * dt * v * Sc;
                    Hpv = dt * mm * (Sc * q) - y1y * dt * Cc;
                    Hpd = dt * mm * (v * Cc * b1 * q) + y1y * dt * v * Sc * b1;
                    Hvd = dt * mm * (Sc * b1 * q) - y1y * dt * Cc * b1 - y1p * c.dtLb * cb * b1;
                    hdd = dt * mm * (v * q * (Cc * b1 * b1 + Sc * b2)) - y1y * dt * v * (-Sc * b1 * b1 + Cc * b2)
                          - y1p * (c.dtLb * v) * (cb * b2 - sb * b1 * b1);
                } else if (u) {
                    const double dt = c.dt;
                    const double e1 = y1x * cs + y1y * sn;
                    const double e2 = y1x * sn - y1y * cs;
                    hpp = dt * sv * e1;
                    Hpv = dt * e2;
                    Hpd = b1 * hpp;
                    Hvd = b1 * Hpv - y1p * c.dtLb * cb * b1;
                    hdd = b1 * b1 * hpp + sv * b2 * Hpv - y1p * (c.dtLb * sv) * (cb * b2 - sb * b1 * b1);
                }
                Recips q;
                recips(k, u, r, sv, ua, ud, rs0, rs1, q);
                const double Sv = zvL * q.vL + zvU * q.vU, bv = mu * (q.vU - q.vL);
                const double Sa = u ? zaL * q.aL + zaU * q.aU : 0.0, ba = u ? mu * (q.aU - q.aL) : 0.0;
                const double Sd = u ? zdL * q.dL + zdU * q.dU : 0.0, bd = u ? mu * (q.dU - q.dL) : 0.0;
                if (r) {
                    SrW0 = rvL0 * q.r0L + rvU0 * q.r0U + dw; br0 = mu * (q.r0U - q.r0L);
                    SrW1 = rvL1 * q.r1L + rvU1 * q.r1U + dw; br1 = mu * (q.r1U - q.r1L);
                    wrow0 = br0 + SrW0 * rdr0;
                    wrow1 = br1 + SrW1 * rdr1;
                }
                Hxx = s2 * wx(k) + dw; Hyy = s2 * wy(k) + dw; Hpp = s2 * wp(k) + hpp + dw; Hvv = s2 * wv(k) + Sv + dw;
                if (MODEL) { Hxx += hss; Hyy += hee; }
                if (u) {
                    if (k >= 1) { Ca = s2 * wt(4); Cd = s2 * wt(5); }
                    if (r) { Ca += SrW1; Cd += SrW0; }
                }
                Haa = u ? s2 * wt(6) + Sa + dw + Ca : 1.0;
                Hdd = u ? s2 * wt(7) + Sd + dw + Cd + hdd : 1.0;
                gsv = g.v + bv;
                if (u) { gua = g.a + ba; gud = g.d + bd; }
            }
            // rate-row terms: +w of the row ending at u_k, -w of the row ending at u_{k+1}
            if (u) {
                gua += wrow1 - ((k + 1 < N) ? wn1 : 0.0);
                gud += wrow0 - ((k + 1 < N) ? wn0 : 0.0);
            }
            double K0[7], K1[7];
            bool pd_ok = true;
            if (!u) {   // terminal cost-to-go
                P[sidx(0, 0)] = Hxx; P[sidx(1, 1)] = Hyy; P[sidx(2, 2)] = Hpp; P[sidx(3, 3)] = Hvv;
                pv[0] = g.x; pv[1] = g.y; pv[2] = g.p; pv[3] = gsv;
            } else if (MODEL) {
                // the s and e_y columns of A are dense and the Hessian has its full 5x5 block: every column of P M, every entry of F
                const double dt = c.dt;
                double Ts[6], Te[6], Tp[6], Tv[6], Ta[6], Td[6], tr[6];
                MPC_UNROLL for (int i = 0; i < 6; i++) {
                    const double p0 = P[sidx(i, 0)], p1 = P[sidx(i, 1)], p2 = P[sidx(i, 2)], p3 = P[sidx(i, 3)], p4 = P[sidx(i, 4)], p5 = P[sidx(i, 5)];
                    Ts[i] = p0 * J.a00 + p2 * J.a20;
                    Te[i] = (p0 * J.a01 + p1) + p2 * J.a21;
                    Tp[i] = (p0 * J.a02 + p1 * J.a12) + p2 * J.a22;
                    Tv[i] = (p0 * J.a03 + p1 * J.a13) + (p2 * J.a23 + p3);
                    Ta[i] = p3 * dt + p4;
                    Td[i] = (p0 * J.b0 + p1 * J.b1) + (p2 * J.b2 + p5);
                    tr[i] = (p0 * r0 + p1 * r1) + (p2 * r2 + p3 * r3 + pv[i]);
                }
                // M' applied to a column T of P M (or to P r + p), row by row of (s, e_y, e_psi, v, a, df)
                auto ms = [&](const double* T) { return J.a00 * T[0] + J.a20 * T[2]; };
                auto me = [&](const double* T) { return (J.a01 * T[0] + T[1]) + J.a21 * T[2]; };
                auto mp = [&](const double* T) { return (J.a02 * T[0] + J.a12 * T[1]) + J.a22 * T[2]; };
                auto mv = [&](const double* T) { return (J.a03 * T[0] + J.a13 * T[1]) + (J.a23 * T[2] + T[3]); };
                auto ma = [&](const double* T) { return T[4] + dt * T[3]; };
                auto md = [&](const double* T) { return (J.b0 * T[0] + J.b1 * T[1] + T[5]) + J.b2 * T[2]; };
                const double Fss = ms(Ts) + Hxx, Fse = ms(Te) + Hse, Fsp = ms(Tp) + Hsp, Fsv = ms(Tv) + Hsv, Fsa = ms(Ta), Fsd = ms(Td) + Hsd;
                const double Fee = me(Te) + Hyy, Fep = me(Tp) + Hep, Fev = me(Tv) + Hev, Fea = me(Ta), Fed = me(Td) + Hed;
                const double Fpp = mp(Tp) + Hpp, Fpv = mp(Tv) + Hpv, Fpa = mp(Ta), Fpd = mp(Td) + Hpd;
                const double Fvv = mv(Tv) + Hvv, Fva = mv(Ta), Fvd = mv(Td) + Hvd;
                const double Faa = ma(Ta) + Haa, Fad = ma(Td);
                const double Fdd = md(Td) + Hdd;
                const double fs = ms(tr) + g.x, fe = me(tr) + g.y, fp = mp(tr) + g.p, fv = mv(tr) + gsv, fa = ma(tr) + gua, fd = md(tr) + gud;
                const double det = Faa * Fdd - Fad * Fad;
                pd_ok = (Faa > 0.0) && (det > 1e-300);
                const double idet = fast_rcp(pd_ok ? det : 1.0);
                const double ja[7] = {Fsa, Fea, Fpa, Fva, -Ca, 0.0, fa}, jd[7] = {Fsd, Fed, Fpd, Fvd, 0.0, -Cd, fd};
                double a0[7], a1[7];
                MPC_UNROLL for (int j = 0; j < 7; j++) {
                    a0[j] = Fdd * ja[j] - Fad * jd[j];
                    a1[j] = Faa * jd[j] - Fad * ja[j];
                    K0[j] = -a0[j] * idet; K1[j] = -a1[j] * idet;
                }
                const double F0[21] = {Fss, Fse, Fsp, Fsv, 0.0, 0.0, Fee, Fep, Fev, 0.0, 0.0, Fpp, Fpv, 0.0, 0.0, Fvv, 0.0, 0.0, Ca, 0.0, Cd};
                MPC_UNROLL for (int i = 0; i < 6; i++)
                    MPC_UNROLL for (int j = i; j < 6; j++) P[sidx(i, j)] = F0[sidx(i, j)] - (ja[i] * a0[j] + jd[i] * a1[j]) * idet;
                const double f0[6] = {fs, fe, fp, fv, 0.0, 0.0};
                MPC_UNROLL for (int i = 0; i < 6; i++) pv[i] = f0[i] - (ja[i] * a0[6] + jd[i] * a1[6]) * idet;
            } else {
                const double A02 = -c.dt * sv * sn, A03 = c.dt * cs, A12 = c.dt * sv * cs, A13 = c.dt * sn, A23 = c.dtLb * sb;
                const double b0 = A02 * b1, b1v = A12 * b1, b2v = c.dtLb * sv * cb * b1, dt = c.dt;
                // columns psi | v | a | df of P M and P r + p  (M = [A B; 0 I], xi = (x, y, psi, v, a_prev, df_prev))
                double Tp[6], Tv[6], Ta[6], Td[6], tr[6];
                MPC_UNROLL for (int i = 0; i < 6; i++) {
                    const double p0 = P[sidx(i, 0)], p1 = P[sidx(i, 1)], p2 = P[sidx(i, 2)], p3 = P[sidx(i, 3)], p4 = P[sidx(i, 4)], p5 = P[sidx(i, 5)];
                    Tp[i] = (p0 * A02 + p1 * A12) + p2;
                    Tv[i] = (p0 * A03 + p1 * A13) + (p2 * A23 + p3);
                    Ta[i] = p3 * dt + p4;
                    Td[i] = (p0 * b0 + p1 * b1v) + (p2 * b2v + p5);
                    tr[i] = (p0 * r0 + p1 * r1) + (p2 * r2 + p3 * r3 + pv[i]);
                }
                // F = H + M' (P M), f = g + M' (P r + p) over (x, y, psi, v, a, df)
                const double Fxx = Hxx + P[sidx(0, 0)], Fxy = P[sidx(0, 1)], Fyy = Hyy + P[sidx(1, 1)];
                const double Fxp = Tp[0], Fxv = Tv[0], Fxa = Ta[0], Fxd = Td[0];
                const double Fyp = Tp[1], Fyv = Tv[1], Fya = Ta[1], Fyd = Td[1];
                const double Fpp = (A02 * Tp[0] + A12 * Tp[1]) + (Tp[2] + Hpp);
                const double Fpv = (A02 * Tv[0] + A12 * Tv[1]) + (Tv[2] + Hpv);
                const double Fpa = (A02 * Ta[0] + A12 * Ta[1]) + Ta[2];
                const double Fpd = (A02 * Td[0] + A12 * Td[1]) + (Td[2] + Hpd);
                const double Fvv = (A03 * Tv[0] + A13 * Tv[1]) + (A23 * Tv[2] + Tv[3] + Hvv);
                const double Fva = (A03 * Ta[0] + A13 * Ta[1]) + (A23 * Ta[2] + Ta[3]);
                const double Fvd = (A03 * Td[0] + A13 * Td[1]) + (A23 * Td[2] + Td[3] + Hvd);
                const double Faa = Ta[4] + (dt * Ta[3] + Haa);
                const double Fad = Td[4] + dt * Td[3];
                const double Fdd = (b0 * Td[0] + b1v * Td[1] + Td[5]) + (b2v * Td[2] + Hdd);
                const double fx = g.x + tr[0], fy = g.y + tr[1];
                const double fp = (A02 * tr[0] + A12 * tr[1]) + (tr[2] + g.p);
                const double fv = (A03 * tr[0] + A13 * tr[1]) + (A23 * tr[2] + tr[3] + gsv);
                const double fa = tr[4] + (dt * tr[3] + gua);
                const double fd = (b0 * tr[0] + b1v * tr[1] + tr[5]) + (b2v * tr[2] + gud);
                // eliminate the inputs: gains K = -Fuu^-1 F_u,xi, cost-to-go P <- F_xixi + F_xi,u K
                const double det = Faa * Fdd - Fad * Fad;
                pd_ok = (Faa > 0.0) && (det > 1e-300);
                const double idet = fast_rcp(pd_ok ? det : 1.0);   // (fast_rcp needs a positive, normal argument)
                const double ja[7] = {Fxa, Fya, Fpa, Fva, -Ca, 0.0, fa}, jd[7] = {Fxd, Fyd, Fpd, Fvd, 0.0, -Cd, fd};
                double a0[7], a1[7];
                MPC_UNROLL for (int j = 0; j < 7; j++) {
                    a0[j] = Fdd * ja[j] - Fad * jd[j];
                    a1[j] = Faa * jd[j] - Fad * ja[j];
                    K0[j] = -a0[j] * idet; K1[j] = -a1[j] * idet;
                }
                const double F0[21] = {Fxx, Fxy, Fxp, Fxv, 0.0, 0.0, Fyy, Fyp, Fyv, 0.0, 0.0, Fpp, Fpv, 0.0, 0.0, Fvv, 0.0, 0.0, Ca, 0.0, Cd};
                MPC_UNROLL for (int i = 0; i < 6; i++)
                    MPC_UNROLL for (int j = i; j < 6; j++) P[sidx(i, j)] = F0[sidx(i, j)] - (ja[i] * a0[j] + jd[i] * a1[j]) * idet;
                const double f0[6] = {fx, fy, fp, fv, 0.0, 0.0};
                MPC_UNROLL for (int i = 0; i < 6; i++) pv[i] = f0[i] - (ja[i] * a0[6] + jd[i] * a1[6]) * idet;
            }
            // ---- stores
            m.sto(TF_GX, k, g.x); m.sto(TF_GY, k, g.y); m.sto(TF_GP, k, g.p); m.sto(TF_GV, k, gsv); m.sto(TF_GA, k, gua); m.sto(TF_GD, k, gud);
            m.sto(TF_HPP, k, Hpp); m.sto(TF_HPV, k, Hpv); m.sto(TF_HVV, k, Hvv); m.sto(TF_HPD, k, Hpd); m.sto(TF_HVD, k, Hvd);
            if (MODEL) {
                m.sto(TF_FH + TFH_SS, k, Hxx); m.sto(TF_FH + TFH_EE, k, Hyy); m.sto(TF_FH + TFH_SE, k, Hse); m.sto(TF_FH + TFH_SP, k, Hsp);
                m.sto(TF_FH + TFH_SV, k, Hsv); m.sto(TF_FH + TFH_SD, k, Hsd); m.sto(TF_FH + TFH_EP, k, Hep); m.sto(TF_FH + TFH_EV, k, Hev);
                m.sto(TF_FH + TFH_ED, k, Hed);
            }
            if (u) {
                m.sto(TF_SRW0, k, SrW0); m.sto(TF_SRW1, k, SrW1); m.sto(TF_BR0, k, br0); m.sto(TF_BR1, k, br1);
                MPC_UNROLL for (int j = 0; j < 7; j++) { m.sto(TF_K + j, k, K0[j]); m.sto(TF_K + 7 + j, k, K1[j]); }
            }
            y1x = yxk; y1y = yyk; y1p = ypk;
            wn0 = wrow0; wn1 = wrow1; na = ua; nd = ud; ua = pa; ud = pd;
            return pd_ok;
        };
        body(N, FalseT{});
        MPC_NOUNROLL for (int k = N - 1; k >= 0; k--) if (!body(k, TrueT{})) return false;
        return true;
    }

    // bound-multiplier steps of stage k from the direction: dz = (mu -/+ z dx) / slack - z
    struct BStep { double vL, vU, aL, aU, dL, dU, r0L, r0U, r1L, r1U; };
    MPC_DEV BStep bound_steps(bool u, bool r, const Recips& q, const double* z, double dsv, double dua, double dud, double drs0, double drs1) const {
        BStep d;
        d.vL = (mu - z[0] * dsv) * q.vL - z[0]; d.vU = (mu + z[1] * dsv) * q.vU - z[1];
        d.aL = d.aU = d.dL = d.dU = d.r0L = d.r0U = d.r1L = d.r1U = 0.0;
        if (u) {
            d.aL = (mu - z[2] * dua) * q.aL - z[2]; d.aU = (mu + z[3] * dua) * q.aU - z[3];
            d.dL = (mu - z[4] * dud) * q.dL - z[4]; d.dU = (mu + z[5] * dud) * q.dU - z[5];
        }
        if (r) {
            d.r0L = (mu - z[6] * drs0) * q.r0L - z[6]; d.r0U = (mu + z[8] * drs0) * q.r0U - z[8];
            d.r1L = (mu - z[7] * drs1) * q.r1L - z[7]; d.r1U = (mu + z[9] * drs1) * q.r1U - z[9];
        }
        return d;
    }
    // order of the TF_Z* fields: vL vU aL aU dL dU rvL0 rvL1 rvU0 rvU1; pairs a stage does not own read as 0
    MPC_DEV void load_z(int k, bool u, bool r, double* z) const {
        z[0] = m.ld(TF_ZVL, k); z[1] = m.ld(TF_ZVU, k);
        MPC_UNROLL for (int i = 2; i < 10; i++) z[i] = 0.0;
        if (u) {
            MPC_UNROLL for (int i = 2; i < 10; i++) z[i] = m.ld(TF_ZVL + i, k);
            if (!r) { z[6] = z[7] = z[8] = z[9] = 0.0; }
        }
    }

    // ------------------------------------------------------------------
    // forward pass (TeamSolver::riccati_forward) + what the line search needs from the direction: slack steps,
    // grad(phi)'d, the tiny-step test, primal and dual fraction-to-the-boundary limits
    // ------------------------------------------------------------------
    MPC_DEV void forward_pass(int rq) {
        const int ec = evb(evcur);
        const bool ls = (rq == 0), soc = (rq == 3);
        const int rb = soc ? TF_C : ec + TEV_RD, db = soc ? TF_C + 4 : ec + TEV_DR;
        double s0 = m.ld(rb + 0, N), s1 = m.ld(rb + 1, N), s2 = m.ld(rb + 2, N), s3 = m.ld(rb + 3, N), pa = 0.0, pd = 0.0;
        if (ls) { s0 = s1 = s2 = s3 = 0.0; }
        double gsum = 0.0;
        bool tl = true;
        const double tt = 10.0 * K_EPS;
        double pnum = 0.0, pden = 1.0, znum = 0.0, zden = 1.0;   // largest ratios by cross-multiplication
        auto body = [&](const int k, auto UT) {
            constexpr bool u = decltype(UT)::value;
            const bool r = u && isR(k);
            if (k + 1 <= N) { m.template prefetch<4>(k + 1, 0, TF_C); m.template prefetch<4>(k + 1, soc ? TF_C : ec, soc ? 6 : TEVN); }
            // ---- loads
            const double sx = m.ld(TF_SX, k), sy = m.ld(TF_SY, k), sp = m.ld(TF_SP, k), sv = m.ld(TF_SV, k);
            const double g0 = m.ld(TF_GX, k), g1 = m.ld(TF_GY, k), g2 = m.ld(TF_GP, k), g3 = m.ld(TF_GV, k);
            double z[10];
            load_z(k, u, r, z);
            double ua = 0.0, ud = 0.0, rs0 = 0.0, rs1 = 0.0, g4 = 0.0, g5 = 0.0;
            double K0[7], K1[7];
            double cs = 0.0, sn = 0.0, cb = 0.0, sb = 0.0, b1 = 0.0, r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0, drr0 = 0.0, drr1 = 0.0;
            double srw0 = 0.0, srw1 = 0.0, brr0 = 0.0, brr1 = 0.0, eq = 0.0, eK = 0.0;
            if (u) {
                ua = m.ld(TF_UA, k); ud = m.ld(TF_UD, k); rs0 = m.ld(TF_RS0, k); rs1 = m.ld(TF_RS1, k);
                g4 = m.ld(TF_GA, k); g5 = m.ld(TF_GD, k);
                MPC_UNROLL for (int j = 0; j < 7; j++) { K0[j] = m.ld(TF_K + j, k); K1[j] = m.ld(TF_K + 7 + j, k); }
                cs = m.ld(ec + TEV_CS, k); sn = m.ld(ec + TEV_SN, k); cb = m.ld(ec + TEV_CB, k); sb = m.ld(ec + TEV_SB, k); b1 = m.ld(ec + TEV_B1, k);
                if (MODEL) { eq = m.ld(ec + TEV_Q, k); eK = m.ld(ec + TEV_K, k); }
                r0 = m.ld(rb + 0, k); r1 = m.ld(rb + 1, k); r2 = m.ld(rb + 2, k); r3 = m.ld(rb + 3, k);
                drr0 = m.ld(db, k); drr1 = m.ld(db + 1, k);
                srw0 = m.ld(TF_SRW0, k); srw1 = m.ld(TF_SRW1, k); brr0 = m.ld(TF_BR0, k); brr1 = m.ld(TF_BR1, k);
                if (ls) { r0 = r1 = r2 = r3 = 0.0; }
                if (ls || !r) { drr0 = drr1 = 0.0; }
                if (!r) { rs0 = rs1 = 0.0; }
            }
            // ---- arithmetic
            double dua = 0.0, dud = 0.0, drs0 = 0.0, drs1 = 0.0;
            double n0 = 0.0, n1 = 0.0, n2 = 0.0, n3 = 0.0;
            if (u) {
                dua = ((K0[4] * pa + K0[5] * pd) + K0[6]) + ((K0[0] * s0 + K0[1] * s1) + (K0[2] * s2 + K0[3] * s3));
                dud = ((K1[4] * pa + K1[5] * pd) + K1[6]) + ((K1[0] * s0 + K1[1] * s1) + (K1[2] * s2 + K1[3] * s3));
                const double A02 = -c.dt * sv * sn, A03 = c.dt * cs, A12 = c.dt * sv * cs, A13 = c.dt * sn, A23 = c.dtLb * sb;
                const double b0 = A02 * b1, b1v = A12 * b1, b2v = c.dtLb * sv * cb * b1;
                n0 = ((s0 + r0) + (A02 * s2 + A03 * s3)) + b0 * dud;
                n1 = ((s1 + r1) + (A12 * s2 + A13 * s3)) + b1v * dud;
                n2 = ((s2 + r2) + A23 * s3) + b2v * dud;
                n3 = (s3 + r3) + c.dt * dua;
                if (MODEL) {   // dense s and e_y columns (TeamSolver::riccati_forward)
                    const FJac J = frenet_jac(cs, sn, cb, sb, b1, eq, eK, sx, sy, sv);
                    n0 = (r0 + (J.a00 * s0 + J.a01 * s1)) + ((J.a02 * s2 + J.a03 * s3) + J.b0 * dud);
                    n1 = ((s1 + r1) + (J.a12 * s2 + J.a13 * s3)) + J.b1 * dud;
                    n2 = (r2 + (J.a20 * s0 + J.a21 * s1)) + ((J.a22 * s2 + J.a23 * s3) + J.b2 * dud);
                }
            }
            double t = g0 * s0 + g1 * s1 + g2 * s2 + g3 * s3 + g4 * dua + g5 * dud;
            if (r) {
                const double bd = (k == 0) ? 0.0 : pd, ba = (k == 0) ? 0.0 : pa;
                drs0 = (dud - bd) + drr0;
                drs1 = (dua - ba) + drr1;
                t += brr0 * drr0 - srw0 * drr0 * (drs0 - drr0);
                t += brr1 * drr1 - srw1 * drr1 * (drs1 - drr1);
            }
            gsum += t;
            tl = tl && fabs(s0) < tt * (1.0 + fabs(sx)) && fabs(s1) < tt * (1.0 + fabs(sy)) && fabs(s2) < tt * (1.0 + fabs(sp)) &&
                 fabs(s3) < tt * (1.0 + fabs(sv)) && fabs(dua) < tt * (1.0 + fabs(ua)) && fabs(dud) < tt * (1.0 + fabs(ud)) &&
                 fabs(drs0) < tt * (1.0 + fabs(rs0)) && fabs(drs1) < tt * (1.0 + fabs(rs1));
            if (!ls) {
                // primal fraction-to-the-boundary: largest -dx / slack, division-free per element
                auto upd = [&](double dx, double sl, double su) {
                    const double n = fabs(dx), d = (dx < 0.0) ? sl : su;
                    if (n * pden > pnum * d) { pnum = n; pden = d; }
                };
                upd(s3, sv - c.vLo, c.vHi - sv);
                if (u) { upd(dua, ua - c.aLo, c.aHi - ua); upd(dud, ud - c.dLo, c.dHi - ud); }
                if (r) { const double h0 = rHi(k, 0), h1 = rHi(k, 1); upd(drs0, rs0 + h0, h0 - rs0); upd(drs1, rs1 + h1, h1 - rs1); }
                // dual fraction-to-the-boundary: largest -dz / z
                Recips q;
                recips(k, u, r, sv, ua, ud, rs0, rs1, q);
                const BStep d = bound_steps(u, r, q, z, s3, dua, dud, drs0, drs1);
                auto lim = [&](double zz, double dz) { if (dz < 0.0 && -dz * zden > znum * zz) { znum = -dz; zden = zz; } };
                lim(z[0], d.vL); lim(z[1], d.vU); lim(z[2], d.aL); lim(z[3], d.aU); lim(z[4], d.dL); lim(z[5], d.dU);
                lim(z[6], d.r0L); lim(z[8], d.r0U); lim(z[7], d.r1L); lim(z[9], d.r1U);
            }
            // ---- stores
            m.sto(TF_DX, k, s0); m.sto(TF_DY, k, s1); m.sto(TF_DP, k, s2); m.sto(TF_DV, k, s3); m.sto(TF_DA, k, dua); m.sto(TF_DD, k, dud);
            m.sto(TF_DRS0, k, drs0); m.sto(TF_DRS1, k, drs1);
            s0 = n0; s1 = n1; s2 = n2; s3 = n3; pa = dua; pd = dud;
        };
        MPC_NOUNROLL for (int k = 0; k < N; k++) body(k, TrueT{});
        body(N, FalseT{});
        p2_gBd = gsum; p2_tiny = tl;
        p2_amax = dmin_(1.0, (pnum > 0.0) ? tau * pden / pnum : 1.0);
        p2_az = dmin_(1.0, (znum > 0.0) ? tau * zden / znum : 1.0);
    }

    // ------------------------------------------------------------------
    // accept pass, backward along the horizon:
    //   costate recursion  lambda_k = l_k + A_k' lambda_{k+1}  (TeamSolver::recover_duals: stationarity in the states)
    //   mode 0: the accepted step: primal, equality multipliers (primal step size), bound multipliers (dual step
    //           size, kappa_sigma safeguard); the trial evaluation becomes the current one
    //   mode 1: least-squares multipliers: y <- lambda
    //   mode 2: nothing is updated
    // and, at the resulting point, the pieces of the optimality error (TeamSolver::solve, PH_BEGIN)
    // ------------------------------------------------------------------
    MPC_DEV void accept_pass(int mode, double al) {
        const int eo = evb(evcur), en = evb(mode == 0 ? (evcur ^ 1) : evcur);
        const double s2 = 2.0 * sigma;
        const bool lsm = ls_system;
        if (mode != 0) al = 0.0;   // (only the accepted step moves the primal point)
        double ny1x = 0.0, ny1y = 0.0, ny1p = 0.0, ny1v = 0.0;            // new multipliers of stage k + 1 (recursion)
        double y1x = 0.0, y1y = 0.0, y1p = 0.0, y1v = 0.0, yd1_0 = 0.0, yd1_1 = 0.0;   // multipliers of stage k + 1 at the resulting point
        double na = 0.0, nd = 0.0;                                       // inputs of stage k + 1 at the resulting point
        double di = 0.0, cv = 0.0, pzabs = 0.0, pzmax = 0.0, pzmin = 1e300, sumy = 0.0, sumz = 0.0, xm = 0.0, ym = 0.0;
        auto body = [&](const int k, auto UT) {
            constexpr bool u = decltype(UT)::value;
            const bool r = u && isR(k);
            if (k >= 1) { m.template prefetch<8>(k - 1, 0, TF_C); m.template prefetch<8>(k - 1, TF_EV, 2 * TEVN + (MODEL ? TFH_N : 0)); }
            // ---- loads
            const int kp = (k >= 1) ? k - 1 : 0;
            double sx = m.ld(TF_SX, k), sy = m.ld(TF_SY, k), sp = m.ld(TF_SP, k), sv = m.ld(TF_SV, k);
            double yx = m.ld(TF_YX, k), yy = m.ld(TF_YY, k), yp = m.ld(TF_YP, k), yv = m.ld(TF_YV, k);
            const double xr = ref(TF_XR, k), yr = ref(TF_YR, k), pr = ref(TF_PR, k);
            const double dsx = m.ld(TF_DX, k), dsy = m.ld(TF_DY, k), dsp = m.ld(TF_DP, k), dsv = m.ld(TF_DV, k);
            const double gx = m.ld(TF_GX, k), gy = m.ld(TF_GY, k), gp = m.ld(TF_GP, k), gv = m.ld(TF_GV, k);
            const double hpp = m.ld(TF_HPP, k), hpv = m.ld(TF_HPV, k), hvv = m.ld(TF_HVV, k), hpd = m.ld(TF_HPD, k), hvd = m.ld(TF_HVD, k);
            const double rd0 = m.ld(en + TEV_RD + 0, k), rd1 = m.ld(en + TEV_RD + 1, k), rd2 = m.ld(en + TEV_RD + 2, k), rd3 = m.ld(en + TEV_RD + 3, k);
            double pa = m.ld(TF_UA, kp), pd = m.ld(TF_UD, kp);   // previous input (not used at k = 0) ...
            const double dpa = m.ld(TF_DA, kp), dpd = m.ld(TF_DD, kp);   // ... and its step
            double z[10];
            load_z(k, u, r, z);
            double ua = 0.0, ud = 0.0, rs0 = 0.0, rs1 = 0.0, ry0 = 0.0, ry1 = 0.0, dua = 0.0, dud = 0.0, drs0 = 0.0, drs1 = 0.0;
            double srw0 = 0.0, srw1 = 0.0, brr0 = 0.0, brr1 = 0.0, dr0 = 0.0, dr1 = 0.0;
            double ocs = 0.0, osn = 0.0, osb = 0.0, ncs = 0.0, nsn = 0.0, ncb = 0.0, nsb = 0.0, nb1 = 0.0;
            double ocb = 0.0, ob1 = 0.0, oq = 0.0, oK = 0.0, nq = 0.0, nK = 0.0;                                  // MODEL 1 only
            double fhss = 0.0, fhee = 0.0, fhse = 0.0, fhsp = 0.0, fhsv = 0.0, fhsd = 0.0, fhep = 0.0, fhev = 0.0, fhed = 0.0;
            if (MODEL) {
                fhss = m.ld(TF_FH + TFH_SS, k); fhee = m.ld(TF_FH + TFH_EE, k); fhse = m.ld(TF_FH + TFH_SE, k); fhsp = m.ld(TF_FH + TFH_SP, k);
                fhsv = m.ld(TF_FH + TFH_SV, k); fhsd = m.ld(TF_FH + TFH_SD, k); fhep = m.ld(TF_FH + TFH_EP, k); fhev = m.ld(TF_FH + TFH_EV, k);
                fhed = m.ld(TF_FH + TFH_ED, k);
            }
            if (u) {
                ua = m.ld(TF_UA, k); ud = m.ld(TF_UD, k); rs0 = m.ld(TF_RS0, k); rs1 = m.ld(TF_RS1, k);
                ry0 = m.ld(TF_RY0, k); ry1 = m.ld(TF_RY1, k);
                dua = m.ld(TF_DA, k); dud = m.ld(TF_DD, k); drs0 = m.ld(TF_DRS0, k); drs1 = m.ld(TF_DRS1, k);
                srw0 = m.ld(TF_SRW0, k); srw1 = m.ld(TF_SRW1, k); brr0 = m.ld(TF_BR0, k); brr1 = m.ld(TF_BR1, k);
                ocs = m.ld(eo + TEV_CS, k); osn = m.ld(eo + TEV_SN, k); osb = m.ld(eo + TEV_SB, k);
                ncs = m.ld(en + TEV_CS, k); nsn = m.ld(en + TEV_SN, k); ncb = m.ld(en + TEV_CB, k); nsb = m.ld(en + TEV_SB, k); nb1 = m.ld(en + TEV_B1, k);
                if (MODEL) {
                    ocb = m.ld(eo + TEV_CB, k); ob1 = m.ld(eo + TEV_B1, k); oq = m.ld(eo + TEV_Q, k); oK = m.ld(eo + TEV_K, k);
                    nq = m.ld(en + TEV_Q, k); nK = m.ld(en + TEV_K, k);
                }
                dr0 = m.ld(en + TEV_DR, k); dr1 = m.ld(en + TEV_DR + 1, k);
                if (!r) { rs0 = rs1 = ry0 = ry1 = drs0 = drs1 = 0.0; }
            }
            // ---- arithmetic
            bool wr_primal = false;
            if (mode != 2) {
                // ---- costates
                const double Hxx = MODEL ? fhss : (lsm ? 1.0 : s2 * wx(k) + dw), Hyy = MODEL ? fhee : (lsm ? 1.0 : s2 * wy(k) + dw);
                double lx = -(Hxx * dsx + gx);
                double ly = -(Hyy * dsy + gy);
                double lp = -(hpp * dsp + hpv * dsv + hpd * dud + gp);
                double lv = -(hpv * dsp + hvv * dsv + hvd * dud + gv);
                if (MODEL) {   // the rest of the 5x5 block (TeamSolver::recover_duals)
                    lx -= fhse * dsy + fhsp * dsp + fhsv * dsv + fhsd * dud;
                    ly -= fhse * dsx + fhep * dsp + fhev * dsv + fhed * dud;
                    lp -= fhsp * dsx + fhep * dsy;
                    lv -= fhsv * dsx + fhev * dsy;
                }
                double nyx = lx + ny1x, nyy = ly + ny1y, nyp = lp + ny1p, nyv = lv + ny1v;
                if (MODEL && u) {   // lambda_k = l_k + A_k' lambda_{k+1} with the dense s and e_y columns, A at the old point
                    const FJac J = frenet_jac(ocs, osn, ocb, osb, ob1, oq, oK, sx, sy, sv);
                    nyx = lx + (J.a00 * ny1x + J.a20 * ny1p);
                    nyy = ly + ((J.a01 * ny1x + ny1y) + J.a21 * ny1p);
                    nyp = lp + ((J.a02 * ny1x + J.a12 * ny1y) + J.a22 * ny1p);
                    nyv = lv + ((J.a03 * ny1x + J.a13 * ny1y) + (J.a23 * ny1p + ny1v));
                } else if (u) {
                    const double A02 = -c.dt * sv * osn, A03 = c.dt * ocs, A12 = c.dt * sv * ocs, A13 = c.dt * osn, A23 = c.dtLb * osb;
                    nyp = (lp + (A02 * ny1x + A12 * ny1y)) + ny1p;
                    nyv = (lv + (A03 * ny1x + A13 * ny1y + A23 * ny1p)) + ny1v;
                }
                double nyd0 = 0.0, nyd1 = 0.0;
                if (r) { nyd0 = srw0 * drs0 + brr0; nyd1 = srw1 * drs1 + brr1; }
                ny1x = nyx; ny1y = nyy; ny1p = nyp; ny1v = nyv;
                if (mode == 1) {
                    double t = dmax_(dmax_(fabs(nyx), fabs(nyy)), dmax_(fabs(nyp), fabs(nyv)));
                    t = dmax_(t, dmax_(fabs(nyd0), fabs(nyd1)));
                    ym = nanmax(ym, t);
                    yx = nyx; yy = nyy; yp = nyp; yv = nyv; ry0 = nyd0; ry1 = nyd1;
                } else {
                    // ---- the accepted step
                    wr_primal = true;
                    Recips q;
                    recips(k, u, r, sv, ua, ud, rs0, rs1, q);
                    const BStep d = bound_steps(u, r, q, z, dsv, dua, dud, drs0, drs1);
                    sx += al * dsx; sy += al * dsy; sp += al * dsp; sv += al * dsv;
                    ua += al * dua; ud += al * dud; rs0 += al * drs0; rs1 += al * drs1;
                    yx += al * (nyx - yx); yy += al * (nyy - yy); yp += al * (nyp - yp); yv += al * (nyv - yv);
                    ry0 += al * (nyd0 - ry0); ry1 += al * (nyd1 - ry1);
                    const double az = p2_az;
                    const double dz[10] = {d.vL, d.vU, d.aL, d.aU, d.dL, d.dU, d.r0L, d.r1L, d.r0U, d.r1U};
                    const double h0 = rHi(k, 0), h1 = rHi(k, 1);
                    const double sl[10] = {sv - c.vLo, c.vHi - sv, ua - c.aLo, c.aHi - ua, ud - c.dLo, c.dHi - ud, rs0 + h0, rs1 + h1, h0 - rs0, h1 - rs1};
                    bool clamp = false;
                    MPC_UNROLL for (int i = 0; i < 10; i++) {
                        const bool own = (i < 2) || (i < 6 ? u : r);
                        if (!own) continue;
                        z[i] += az * dz[i];
                        const double pz = z[i] * sl[i];
                        clamp = clamp || (pz > K_KAPPA_SIGMA * mu) || (pz * K_KAPPA_SIGMA < mu);
                    }
                    if (clamp) kappa_sigma_clamp(z, sl, mu);
                }
            }
            // ---- optimality error pieces at the resulting point.  The objective gradient needs the previous input at the
            // resulting point, which this backward pass has not reached yet: it is formed from the old value and its step.
            pa += al * dpa; pd += al * dpd;
            Grad g;
            {
                g.x = s2 * wx(k) * (sx - xr); g.y = s2 * wy(k) * (sy - yr); g.p = s2 * wp(k) * (sp - pr); g.v = s2 * wv(k) * (sv - cst[6]);
                g.a = 0.0; g.d = 0.0;
                if (u) {
                    g.a = s2 * wt(6) * ua;
                    g.d = s2 * wt(7) * ud;
                    if (k >= 1) { g.a += s2 * wt(4) * (ua - pa); g.d += s2 * wt(5) * (ud - pd); }
                    if (k + 1 < N) { g.a -= s2 * wt(4) * (na - ua); g.d -= s2 * wt(5) * (nd - ud); }
                }
            }
            const double hn = u ? 1.0 : 0.0;
            double A02 = 0.0, A03 = 0.0, A12 = 0.0, A13 = 0.0, A23 = 0.0, b0 = 0.0, b1v = 0.0, b2v = 0.0;
            if (u) {
                A02 = -c.dt * sv * nsn; A03 = c.dt * ncs; A12 = c.dt * sv * ncs; A13 = c.dt * nsn; A23 = c.dtLb * nsb;
                b0 = A02 * nb1; b1v = A12 * nb1; b2v = c.dtLb * sv * ncb * nb1;
            }
            double glx = g.x + yx - hn * y1x;
            double gly = g.y + yy - hn * y1y;
            double glp = g.p + yp - hn * (A02 * y1x + A12 * y1y + y1p);
            double glv = g.v + yv - hn * (A03 * y1x + A13 * y1y + A23 * y1p + y1v) - z[0] + z[1];
            double jd = b0 * y1x + b1v * y1y + b2v * y1p;
            if (MODEL && u) {   // the stage Jacobian of the Frenet map at the resulting point
                const FJac J = frenet_jac(ncs, nsn, ncb, nsb, nb1, nq, nK, sx, sy, sv);
                glx = g.x + yx - (J.a00 * y1x + J.a20 * y1p);
                gly = g.y + yy - (J.a01 * y1x + hn * y1y + J.a21 * y1p);
                glp = g.p + yp - (J.a02 * y1x + J.a12 * y1y + J.a22 * y1p);
                glv = g.v + yv - (J.a03 * y1x + J.a13 * y1y + J.a23 * y1p + hn * y1v) - z[0] + z[1];
                jd = J.b0 * y1x + J.b1 * y1y + J.b2 * y1p;
            }
            const double nd0 = (k + 1 < N) ? yd1_0 : 0.0, nd1 = (k + 1 < N) ? yd1_1 : 0.0;
            const double gla = g.a - hn * c.dt * y1v + (ry1 - nd1) - z[2] + z[3];
            const double gld = g.d - hn * jd + (ry0 - nd0) - z[4] + z[5];
            double t = dmax_(dmax_(fabs(glx), fabs(gly)), dmax_(fabs(glp), fabs(glv)));
            t = dmax_(t, dmax_(fabs(gla), fabs(gld)));
            t = dmax_(t, dmax_(fabs(-ry0 - z[6] + z[8]), fabs(-ry1 - z[7] + z[9])));
            di = nanmax(di, t);
            double cvk = dmax_(dmax_(fabs(rd0), fabs(rd1)), dmax_(fabs(rd2), fabs(rd3)));
            cvk = dmax_(cvk, dmax_(fabs(dr0), fabs(dr1)));
            cv = nanmax(cv, cvk);
            sumy += fabs(yx) + fabs(yy) + fabs(yp) + fabs(yv) + fabs(ry0) + fabs(ry1);
            sumz += z[0] + z[1] + z[2] + z[3] + z[4] + z[5] + z[6] + z[7] + z[8] + z[9];
            {   // complementarity products of the owned bound pairs
                const double h0 = rHi(k, 0), h1 = rHi(k, 1);
                const double sl[10] = {sv - c.vLo, c.vHi - sv, ua - c.aLo, c.aHi - ua, ud - c.dLo, c.dHi - ud, rs0 + h0, rs1 + h1, h0 - rs0, h1 - rs1};
                MPC_UNROLL for (int i = 0; i < 10; i++) {
                    const bool own = (i < 2) || (i < 6 ? u : r);
                    if (!own) continue;
                    const double pz = sl[i] * z[i];
                    pzabs = nanmax(pzabs, fabs(pz)); pzmax = nanmax(pzmax, pz); pzmin = (pz < pzmin || pz != pz) ? pz : pzmin;
                }
            }
            xm = nanmax(xm, dmax_(dmax_(fabs(sx), fabs(sy)), dmax_(fabs(sp), fabs(sv))));
            // ---- stores
            if (wr_primal) {
                m.sto(TF_SX, k, sx); m.sto(TF_SY, k, sy); m.sto(TF_SP, k, sp); m.sto(TF_SV, k, sv);
                m.sto(TF_ZVL, k, z[0]); m.sto(TF_ZVU, k, z[1]);
                if (u) {
                    m.sto(TF_UA, k, ua); m.sto(TF_UD, k, ud);
                    MPC_UNROLL for (int i = 2; i < 6; i++) m.sto(TF_ZVL + i, k, z[i]);
                }
                if (r) {
                    m.sto(TF_RS0, k, rs0); m.sto(TF_RS1, k, rs1);
                    MPC_UNROLL for (int i = 6; i < 10; i++) m.sto(TF_ZVL + i, k, z[i]);
                }
            }
            if (mode != 2) {
                m.sto(TF_YX, k, yx); m.sto(TF_YY, k, yy); m.sto(TF_YP, k, yp); m.sto(TF_YV, k, yv);
                if (r) { m.sto(TF_RY0, k, ry0); m.sto(TF_RY1, k, ry1); }
            }
            y1x = yx; y1y = yy; y1p = yp; y1v = yv; yd1_0 = ry0; yd1_1 = ry1; na = ua; nd = ud;
        };
        body(N, FalseT{});
        MPC_NOUNROLL for (int k = N - 1; k >= 0; k--) body(k, TrueT{});
        e_di = di; e_cv = cv; e_pzabs = pzabs; e_pzmax = pzmax; e_pzmin = pzmin; e_sumy = sumy; e_sumz = sumz; e_xm = xm; e_ym = ym;
        if (mode == 0) evcur ^= 1;
    }

    MPC_DEV void zero_multipliers() {
        for (int k = 0; k <= N; k++) {
            m.sto(TF_YX, k, 0.0); m.sto(TF_YY, k, 0.0); m.sto(TF_YP, k, 0.0); m.sto(TF_YV, k, 0.0);
            m.sto(TF_RY0, k, 0.0); m.sto(TF_RY1, k, 0.0);
        }
    }

    // c_soc <- a_soc c_soc + c(trial)  (first correction: c_soc = the residuals at the current point)
    MPC_DEV void soc_accumulate(bool first, double as) {
        const int ec = evb(evcur), et = evb(evcur ^ 1);
        for (int k = 0; k <= N; k++) {
            for (int i = 0; i < 4; i++) {
                const double old = first ? m.ld(ec + TEV_RD + i, k) : m.ld(TF_C + i, k);
                m.sto(TF_C + i, k, as * old + m.ld(et + TEV_RD + i, k));
            }
            if (isU(k)) for (int i = 0; i < 2; i++) {
                const double old = first ? m.ld(ec + TEV_DR + i, k) : m.ld(TF_C + 4 + i, k);
                m.sto(TF_C + 4 + i, k, as * old + m.ld(et + TEV_DR + i, k));
            }
        }
    }

    // restoration by rollout (TeamSolver::rollout_restore / rollout_core): the iterate's inputs projected stage by
    // stage onto the input box, the rate rows and the speed bounds; states rolled out from the measured state
    MPC_DEV void rollout_restore() {
        double s0 = cst[0], s1 = cst[1], s2 = cst[2], s3 = cst[3];
        double pa = cst[5], pd = cst[4];
        for (int s = 0; s < N; s++) {
            double ua = m.ld(TF_UA, s), ud = m.ld(TF_UD, s);
            if (s != 1) {
                const double h = (s == 0) ? c.dtc : c.dt;
                const double la = 0.98 * c.admax * h, ld = 0.98 * c.sdmax * h;
                ua = dmin_(dmax_(ua, pa - la), pa + la);
                ud = dmin_(dmax_(ud, pd - ld), pd + ld);
            }
            ua = dmin_(dmax_(ua, -c.amax), c.amax);
            ud = dmin_(dmax_(ud, -c.smax), c.smax);
            ua = dmin_(dmax_(ua, (c.vmin - s3) / c.dt), (c.vmax - s3) / c.dt);
            m.sto(TF_SX, s, s0); m.sto(TF_SY, s, s1); m.sto(TF_SP, s, s2); m.sto(TF_SV, s, s3); m.sto(TF_UA, s, ua); m.sto(TF_UD, s, ud);
            double sd, cd, sps, cps;
            mpc_sincos(ud, &sd, &cd);
            mpc_sincos(s2, &sps, &cps);
            const double rr = c.rfrac;
            const double inv = sqrt(1.0 / (cd * cd + rr * rr * sd * sd));
            const double cb = cd * inv, sb = rr * sd * inv;
            double n0 = s0 + c.dt * (s3 * (cps * cb - sps * sb));
            const double n1 = s1 + c.dt * (s3 * (sps * cb + cps * sb));
            double n2 = s2 + c.dtLb * (s3 * sb);
            const double n3 = s3 + c.dt * ua;
            if (MODEL) {   // Frenet frame (MKZMPCPathFollowerFrenet.jl:111-120): (s, e_y, e_psi, v)
                const double K = curvature(s0).K;
                const double g = s3 * (cps * cb - sps * sb) / (1.0 - s1 * K);
                n0 = s0 + c.dt * g;
                n2 = s2 + (c.dtLb * (s3 * sb) - c.dt * (g * K));
            }
            s0 = n0; s1 = n1; s2 = n2; s3 = n3; pa = ua; pd = ud;
        }
        m.sto(TF_SX, N, s0); m.sto(TF_SY, N, s1); m.sto(TF_SP, N, s2); m.sto(TF_SV, N, s3); m.sto(TF_UA, N, 0.0); m.sto(TF_UD, N, 0.0);
    }

    MPC_DEV bool filter_ok(double ph_t, double th_t) const {
        for (int e = 0; e < nfilt; e++) {
            const double fp = m.fld(2 * e), ft = m.fld(2 * e + 1);
            if (!(cmp_le(ph_t, fp, fp) || cmp_le(th_t, ft, ft))) return false;
        }
        return true;
    }
    MPC_DEV void filter_add(double fp, double ft) {
        if (nfilt < TPP_NFILT) {
            m.fst(2 * nfilt, fp); m.fst(2 * nfilt + 1, ft);
            nfilt++;
        }
    }

    // ------------------------------------------------------------------
    // One trip.  Every pass along the horizon has exactly ONE call site, in a fixed order, so that lanes that are in
    // different iterations (or different problems) run the same instruction stream and the kernel stays small:
    //     [rare: restoration / interior start / second-order-correction right-hand side]
    //     [backward + forward]  after_solve()   [trial]  after_eval()   [accept]  after_accept()
    // `op` says which section a lane enters next; a section that does not match is skipped until the next trip.
    // The three driver pieces are TeamSolver::solve's phase machine cut at the points where it asks for a pass.
    // Returns true when the solve has ended.
    // ------------------------------------------------------------------
    enum { OP_SOLVE = 0, OP_EVAL, OP_ACCEPT, OP_INIT, OP_RESTO, OP_SOC_ACC, OP_ZERO_Y };
    // All the warps of a block enter each section together (block barrier): at any time an SM then runs ONE stage body,
    // which its instruction cache holds, instead of eight warps spread over the whole kernel (measured: instruction-fetch
    // stalls were the largest stall reason without the barriers).  Every thread of the block calls tick() on every
    // trip, lanes without a running problem with live = false.
    MPC_DEV static void pass_sync() {
#if !defined(MPC_HOST_EMU) && !defined(MPC_TPP_NO_PASS_SYNC)
        __syncthreads();
#endif
    }
    MPC_DEV bool tick(bool live) {
        if (live && ret != RUNNING) live = false;
        pass_sync();
        if (live && op >= OP_INIT) {
            if (op == OP_SOC_ACC) { soc_accumulate(soc_first, a_soc); op = OP_SOLVE; req = 3; }
            else if (op == OP_ZERO_Y) { zero_multipliers(); op = OP_ACCEPT; acc_mode = 2; }
            else {
                if (op == OP_RESTO) { rollout_restore(); zero_multipliers(); }
                init_pass();
                phase = PH_EVAL0; op = OP_EVAL; ev_alpha = 0.0;
            }
        }
        pass_sync();
        if (live && op == OP_SOLVE) {
            ls_system = (req == 0);
            solve_ok = backward_pass(req);
        }
        pass_sync();
        if (live && op == OP_SOLVE) {
            if (solve_ok) forward_pass(req);
            after_solve();
        }
        pass_sync();
        if (live && ret == RUNNING && op == OP_EVAL) {
            eval_pass(ev_alpha);
            after_eval();
        }
        pass_sync();
        if (live && ret == RUNNING && op == OP_ACCEPT) {
            accept_pass(acc_mode, alpha);
            after_accept();
        }
        return ret != RUNNING;
    }

    // line search cannot go on from the current point (Ipopt would enter the restoration phase)
    MPC_DEV void line_search_failed() {
        if (cur_acceptable) { ret = 1; return; }   // ... unless the point is acceptable: Solved_To_Acceptable_Level
        if (cur_theta <= 1e-2 * c.tol) { ret = had_acceptable ? 1 : -2; return; }   // ... or almost feasible
        if (n_resto < K_MAX_RESTO) {
            n_resto++; had_acceptable = false;
            filter_add(phi - K_GAMMA_PHI * cur_theta, (1.0 - K_GAMMA_THETA) * cur_theta);   // the point that is left enters the filter
            resto_check = true; tiny_last = false;
            iter++;
            op = OP_RESTO;
            return;
        }
        ret = -2;
    }

    MPC_DEV void after_solve() {
        if (phase == PH_LS) {   // least-squares multipliers: taken if the solve went through (their size is checked after the pass)
            op = OP_ACCEPT; acc_mode = solve_ok ? 1 : 2;
            return;
        }
        if (phase == PH_SOC) {   // second-order correction: straight on to its trial point
            ev_alpha = p2_amax; a_soc = ev_alpha;
            op = OP_EVAL;
            return;
        }
        // PH_PD, PH_RESOLVE
        if (!solve_ok) {
            // PDPerturbationHandler::PerturbForWrongInertia
            if (dw == 0.0) dw = (dw_last == 0.0) ? K_DW_INIT : dmax_(K_DW_MIN, dw_last * K_DW_DEC);
            else dw = (dw_last == 0.0 || 1e5 * dw_last < dw) ? K_DW_INC_FIRST * dw : K_DW_INC * dw;
            if (dw > K_DW_MAX) { ret = -4; return; }
            req = 2;   // op stays OP_SOLVE: next trip
            return;
        }
        if (phase == PH_RESOLVE) {
            alpha = alpha_max * 0.5; nsteps = 1;
            double alpha_min = K_GAMMA_THETA;
            if (gBd < 0.0) alpha_min = dmin_(K_GAMMA_THETA, K_GAMMA_PHI * cur_theta / (-gBd));
            bool above_min = alpha > alpha_min * K_ALPHA_MIN_FRAC;
            if (!above_min && gBd < 0.0 && cur_theta <= theta_min)
                above_min = ratio_test(1, alpha, K_ALPHA_MIN_FRAC * (K_DELTA * Rft), cur_theta, -gBd);
            if (!above_min) { line_search_failed(); return; }
            ev_alpha = alpha; op = OP_EVAL; phase = PH_TRIAL;
            return;
        }
        if (dw > 0.0) dw_last = dw;
        // ---- line-search quantities at the current point
        const double theta = cur_theta;
        phi = sigma * cur_f - mu * cur_lb;
        gBd = p2_gBd;
        tiny = p2_tiny && (theta < 1e-4);
        if (theta_max < 0.0) { theta_max = 1e4 * dmax_(1.0, theta); theta_min = 1e-4 * dmax_(1.0, theta); }
        // switching-condition ratio theta^s_theta / (-gBd)^s_phi, single-precision estimate (see ratio_test)
        Rft = (gBd < 0.0) ? (double)fast_exp2((float)K_S_THETA * fast_log2((float)theta) - (float)K_S_PHI * fast_log2((float)(-gBd))) : 0.0;
        alpha_max = p2_amax;
        alpha = alpha_max; nsteps = 0;
        ev_alpha = alpha; op = OP_EVAL; phase = PH_TRIAL;
    }

    MPC_DEV void after_eval() {
        if (phase == PH_EVAL0) {
            evcur ^= 1;   // the evaluation just made is the current point's
            if (resto_check) {   // the restored point must be acceptable to the filter
                const double th_r = ev_theta, ph_r = sigma * ev_f - mu * ev_lb;
                bool ok = (th_r == th_r) && (ph_r == ph_r) && cmp_le(th_r, theta_max, theta_max);
                ok = filter_ok(ph_r, th_r) && ok;
                if (!ok) { ret = -2; return; }
                resto_check = false;
            }
            cur_theta = ev_theta; cur_f = ev_f; cur_lb = ev_lb;
            phase = PH_LS; op = OP_SOLVE; req = 0;
            return;
        }
        // PH_TRIAL, PH_SOC
        const double alpha_test = (phase == PH_SOC) ? alpha_max : alpha;
        const double th_t = ev_theta;
        const double ph_t = sigma * ev_f - mu * ev_lb;
        const double theta = cur_theta;
        const bool ftype = (gBd < 0.0) && ratio_test(0, alpha_test, K_DELTA * Rft, theta, -gBd);
        const bool arm = cmp_le(ph_t - phi, K_ETA_PHI * alpha_test * gBd, phi);
        bool ok = tiny;
        if (!tiny) {
            ok = (th_t == th_t) && (ph_t == ph_t);
            if (ok && !cmp_le(th_t, theta_max, theta)) ok = false;
            if (ok) {
                if (ftype && theta <= theta_min) ok = arm;
                else {
                    if (ph_t > phi) {
                        double bas = 1.0; if (fabs(phi) > 10.0) bas = log10(fabs(phi));
                        if (log10(ph_t - phi) > K_OBJ_MAX_INC + bas) ok = false;
                    }
                    if (ok) ok = cmp_le(th_t, (1.0 - K_GAMMA_THETA) * theta, theta) || cmp_le(ph_t - phi, -K_GAMMA_PHI * theta, phi);
                }
            }
            ok = filter_ok(ph_t, th_t) && ok;
        }
        if (!ok) {
            bool want_soc = false;
            if (phase == PH_TRIAL) {
                if (nsteps == 0 && theta <= th_t && K_MAX_SOC > 0) { want_soc = true; soc_cnt = 0; a_soc = alpha; }
            } else {
                soc_cnt++;
                want_soc = (soc_cnt < K_MAX_SOC) && (th_t <= K_KAPPA_SOC * th_soc_old);
            }
            if (want_soc) {
                // c_soc <- a_soc * c_soc + c(trial), then the same matrix with that right-hand side
                th_soc_old = th_t;
                soc_first = (phase == PH_TRIAL);
                phase = PH_SOC; op = OP_SOC_ACC;
                return;
            }
            if (phase == PH_SOC) {
                // corrections exhausted: recompute the Newton direction (the current evaluation was kept), backtrack
                phase = PH_RESOLVE; op = OP_SOLVE; req = 1;
                return;
            }
            // plain backtracking
            double alpha_min = K_GAMMA_THETA;
            if (gBd < 0.0) alpha_min = dmin_(K_GAMMA_THETA, K_GAMMA_PHI * theta / (-gBd));
            alpha_min *= K_ALPHA_MIN_FRAC;
            alpha *= 0.5; nsteps++;
            bool above_min = alpha > alpha_min;
            if (!above_min && gBd < 0.0 && theta <= theta_min)
                above_min = ratio_test(1, alpha, K_ALPHA_MIN_FRAC * (K_DELTA * Rft), theta, -gBd);
            if (!above_min) { line_search_failed(); return; }
            ev_alpha = alpha; phase = PH_TRIAL;   // op stays OP_EVAL: next trip
            return;
        }
        // ---------------- accepted ----------------
        if (phase == PH_SOC) alpha = a_soc;
        if (!tiny && !(ftype && arm)) filter_add(phi - K_GAMMA_PHI * theta, (1.0 - K_GAMMA_THETA) * theta);
        op = OP_ACCEPT; acc_mode = 0;
    }

    MPC_DEV void after_accept() {
        const int nz = 2 * (3 * N + 1) + 4 * (N - 1);  // bound multipliers: x-bounds + slack bounds
        const int my = 4 * (N + 1) + 2 * (N - 1);      // equality multipliers y_c, y_d
        if (acc_mode == 0) {
            // the accepted trial evaluation is the next iteration's current evaluation
            cur_theta = ev_theta; cur_f = ev_f; cur_lb = ev_lb;
            tiny_last = tiny;
            iter++;
        } else if (acc_mode == 1 && !(e_ym <= K_Y_INIT_MAX)) {   // least-squares multipliers too large: start from zero
            op = OP_ZERO_Y;
            return;
        }
        // ---- PH_BEGIN: optimality error at the current point, convergence, barrier update
        const double sumy = e_sumy, sumz = e_sumz;
        const double sty = sumy + sumz;
        const bool big_d = sty > K_S_MAX * (double)(my + nz), big_c = sumz > K_S_MAX * (double)nz;
        double sd = 1.0, sc = 1.0;
        if (big_d) sd = div_cold(sty, (double)(my + nz) * K_S_MAX);
        if (big_c) sc = div_cold(sumz, (double)nz * K_S_MAX);
        const double cm0 = e_pzabs;
        const double cmm = dmax_(fabs(e_pzmax - mu), fabs(e_pzmin - mu));
        const double dcv = dmax_(big_d ? div_cold(e_di, sd) : e_di, e_cv);
        const double e0 = dmax_(dcv, big_c ? div_cold(cm0, sc) : cm0);
        double em = dmax_(dcv, big_c ? div_cold(cmm, sc) : cmm);
        // ---- convergence (OptimalityErrorConvergenceCheck)
        if (e0 <= dmax_(K_ACCEPT_TOL, c.tol)) {
            const double du = e_di / sigma, cvm = e_cv, mc = cm0 / sigma;
            if (e0 <= c.tol && du <= 1.0 && cvm <= 1e-4 && mc <= 1e-4) { ret = 0; return; }
            cur_acceptable = (e0 <= K_ACCEPT_TOL && du <= 1e10 && cvm <= 1e-2 && mc <= 1e-2);
            if (cur_acceptable) { had_acceptable = true; if (++accept_count >= K_ACCEPT_ITER) { ret = 1; return; } }
            else accept_count = 0;
        } else { accept_count = 0; cur_acceptable = false; }
        if (iter >= c.max_iter) { ret = -1; return; }
        if (!(e_xm <= 1e20)) { ret = -5; return; }
        // ---- monotone barrier update
        for (;;) {
            if (!(em <= K_KAPPA_EPS * mu) && !tiny_last) break;
            const double nm = dmax_(c.mu_min, dmin_(K_KAPPA_MU * mu, mu * sqrt(mu)));
            if (nm >= mu) { if (tiny_last) ret = -3; break; }
            mu = nm; tau = dmax_(K_TAU_MIN, 1.0 - mu);
            nfilt = 0;
            if (tiny_last) { tiny_last = false; break; }
            const double cl = dmax_(fabs(e_pzmax - mu), fabs(e_pzmin - mu));
            em = dmax_(dcv, big_c ? div_cold(cl, sc) : cl);
        }
        if (ret == -3) return;
        dw = 0.0;
        phase = PH_PD; op = OP_SOLVE; req = 1;
    }

    // ------------------------------------------------------------------
    // results (solve_problem's epilogue): status, honor_original_bounds, unscaled objective, outputs
    // ------------------------------------------------------------------
    MPC_DEV void finish(const BatchPtrs& io, long b) {
        const long nt = 6L * N + 4;
        const int status = (ret == 0 || ret == 1) ? 0 : (ret == 2 ? 1 : (ret == -1 ? 3 : (ret == -5 ? 2 : 4)));
        double* t0 = io.traj ? io.traj + nt * b : nullptr;
        double* t1 = io.warm ? io.warm + nt * b : nullptr;
        double f = 0.0, pa = 0.0, pd = 0.0, a0 = 0.0, d0 = 0.0;
        for (int k = 0; k <= N; k++) {
            const double sx = m.ld(TF_SX, k), sy = m.ld(TF_SY, k), sp = m.ld(TF_SP, k);
            double sv = m.ld(TF_SV, k), ua = isU(k) ? m.ld(TF_UA, k) : 0.0, ud = isU(k) ? m.ld(TF_UD, k) : 0.0;
            if (feasible) {
                sv = dmin_(dmax_(sv, c.vmin), c.vmax);
                if (isU(k)) { ua = dmin_(dmax_(ua, -c.amax), c.amax); ud = dmin_(dmax_(ud, -c.smax), c.smax); }
            }
            const double ex = sx - ref(TF_XR, k), ey = sy - ref(TF_YR, k), ep = sp - ref(TF_PR, k), evv = sv - cst[6];
            double fk = wx(k) * ex * ex + wy(k) * ey * ey + wp(k) * ep * ep + wv(k) * evv * evv;
            if (isU(k)) {
                fk += wt(6) * ua * ua + wt(7) * ud * ud;
                if (k >= 1) { const double da = ua - pa, dd = ud - pd; fk += wt(4) * da * da + wt(5) * dd * dd; }
            }
            f += fk;
            if (k == 0) { a0 = ua; d0 = ud; }
            for (int pass = 0; pass < 2; pass++) {
                double* t = pass ? t1 : t0;
                if (!t) continue;
                t[k] = sx; t[(N + 1) + k] = sy; t[2 * (N + 1) + k] = sv; t[3 * (N + 1) + k] = sp;
                if (isU(k)) { t[4 * (N + 1) + k] = ud; t[4 * (N + 1) + N + k] = ua; }
            }
            pa = ua; pd = ud;
        }
        if (io.u0) { io.u0[2 * b] = a0; io.u0[2 * b + 1] = d0; }
        if (io.cost) io.cost[b] = f;
        if (io.status) io.status[b] = status;
        if (io.iters) io.iters[b] = iter;
        if (io.rec) { st_global_v2(io.rec + 4 * b, a0, d0); st_global_v2(io.rec + 4 * b + 2, f, int2_as_double(status | (n_resto << 8), iter)); }
        if (io.resto) io.resto[b] = n_resto;
    }
};
typedef TppSolverT<0> TppSolver;

}  // namespace mpcb200
