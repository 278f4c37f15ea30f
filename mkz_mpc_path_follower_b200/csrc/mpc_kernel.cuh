// mpc_kernel.cuh -- one MPC problem per warp (or per block of 2-3 warps): interior-point iteration
// with a Riccati KKT solve.
//
// What it replaces (reference file:line):
//   NLP transcription   scripts/mpc_utils/MKZMPCPathFollower.jl:65-123  (JuMP AD -> analytic
//                       stage Jacobians A_k, B_k and the (psi,v,df) Lagrangian-Hessian block)
//   solve(mdl)          scripts/mpc_utils/MKZMPCPathFollower.jl:176      (Ipopt: barrier update,
//                       fraction-to-boundary, filter line search, inertia correction; MUMPS LDL^T
//                       -> block-tridiagonal Riccati recursion on the condensed KKT system)
//
// Thread k of a TEAM owns stage k of the horizon (k = 0..N).  A team is one warp for N <= 31 (the
// hot configuration: four independent problems per block) and one block of W = 2 or 3 warps for
// long horizons (N <= 63 / 95: one problem per block; cross-warp exchanges go through a small
// shared-memory area and bar.sync, the serial Riccati recursion runs in warp 0).  Thread k holds
// its state (x,y,psi,v), input (acc,df), the multipliers of the equality rows that define s_k, its
// bound multipliers and the rate row that ends at u_k.  Stage-parallel work (model evaluation,
// residuals, multiplier updates, norms) runs with threads = stages; the serial Riccati recursion
// switches to lanes = matrix entries, with per-stage records staged in shared memory.
//
// The iteration follows oracle/mpc_oracle.c step for step (same formulas, same constants);
// only the linear algebra differs (condensed Riccati here, full-space Bunch-Kaufman there).
// Ipopt's restoration phase is not restated: a failed line search is answered by a restoration by
// rollout (rollout_restore), the same in both implementations.
//
// Control flow is a warp-uniform phase machine so that every heavy routine (record assembly,
// Riccati backward/forward, dual recovery, trial-point evaluation) exists exactly once in the
// instruction stream: least-squares multiplier solve, Newton solves with inertia-correction
// retries, second-order corrections and line-search trials all pass through the same code.
// The phase machine makes all solver state look live everywhere, so only the primal iterate and the
// equality multipliers stay in registers; bound multipliers, step, model evaluation and reference
// sample live in per-thread shared-memory fields (LF_*): 168 registers, 12 warps per SM at N = 20.
//
// MODEL template parameter: 0 = the XY model above; 1 = the reference's Frenet-frame variant
// (scripts/mpc_utils/MKZMPCPathFollowerFrenet.jl:65-123: states s, e_y, e_psi, v in the slots of x, y, psi, v;
// ds/dt = v cos(e_psi + beta) / (1 - e_y K(s)), K a cubic per problem).  Same driver, bounds, rate rows and cost form;
// the `if (MODEL)` branches hold what differs: the stage map and its 5x5 Lagrangian-Hessian block (eval_point,
// frenet_jac, assemble), two more columns of P M in Riccati round A, the dense forward sweep and a serial costate
// recursion in place of the suffix sums (recover_duals).  The XY instantiation compiles to the same code as before.
#pragma once
#include "warp_prims.cuh"
#ifdef MPC_TRACE
#include <cstdio>
#endif

namespace mpcb200 {

#ifdef MPC_HOST_EMU
#define MPC_HD inline
#define MPC_NOUNROLL
#else
#define MPC_HD __host__ __device__ __forceinline__
#define MPC_NOUNROLL _Pragma("unroll 1")
#endif

struct KCfg {
    int N, max_iter, start_mode, pad_;
    double dt, dtc, La, Lb, vmin, vmax, amax, smax, admax, sdmax, tol;
    double w[8];  // cx, cy, cpsi, cv, cdacc, cddf, cacc, cdf
    // derived on the host by kcfg_finalize(): bounds relaxed by Ipopt's bound_relax_factor etc.
    double vLo, vHi, aLo, aHi, dLo, dHi;
    double rHiFirst[2], rHiLater[2];  // relaxed half-width of the rate rows [steer, acc]; rLo = -rHi
    double rfrac;                     // L_b / (L_a + L_b)
    double mu_min;
    double dtLb;                      // dt / L_b (multiplying by it avoids a division per use; 0 / x takes the slow division path)
    const int* roles;                 // [32][ROLE_STRIDE] lane roles of the Riccati recursion (riccati_roles), device memory
};

// ---- Ipopt 3.12 default constants (same values as oracle/mpc_oracle.c) ----
#define K_KAPPA_EPS 10.0
#define K_KAPPA_MU 0.2
#define K_MU_INIT 0.1
#define K_TAU_MIN 0.99
#define K_BOUND_PUSH 1e-2
#define K_BOUND_FRAC 1e-2
#define K_BOUND_RELAX 1e-8
#define K_S_MAX 100.0
#define K_KAPPA_SIGMA 1e10
#define K_GAMMA_THETA 1e-5
#define K_GAMMA_PHI 1e-8
#define K_ETA_PHI 1e-8
#define K_DELTA 1.0
#define K_S_THETA 1.1
#define K_S_PHI 2.3
#define K_ALPHA_MIN_FRAC 0.05
#define K_MAX_SOC 4
#define K_KAPPA_SOC 0.99
#define K_OBJ_MAX_INC 5.0
#define K_DW_INIT 1e-4
#define K_DW_MIN 1e-20
#define K_DW_MAX 1e20
#define K_DW_INC_FIRST 100.0
#define K_DW_INC 8.0
#define K_DW_DEC (1.0 / 3.0)
#define K_SCALE_MAX_GRAD 100.0
#define K_Y_INIT_MAX 1e3
#define K_ACCEPT_TOL 1e-6
#define K_ACCEPT_ITER 15
#define K_MAX_RESTO 3      // restorations by rollout per solve (not an Ipopt option; see rollout_restore)
#define K_EPS 2.220446049250313e-16

MPC_HD void kcfg_finalize(KCfg& c) {
    auto mx = [](double a, double b) { return a > b ? a : b; };
    auto ab = [](double a) { return a < 0 ? -a : a; };
    c.vLo = c.vmin - K_BOUND_RELAX * mx(1.0, ab(c.vmin)); c.vHi = c.vmax + K_BOUND_RELAX * mx(1.0, ab(c.vmax));
    c.aLo = -c.amax - K_BOUND_RELAX * mx(1.0, c.amax); c.aHi = c.amax + K_BOUND_RELAX * mx(1.0, c.amax);
    c.dLo = -c.smax - K_BOUND_RELAX * mx(1.0, c.smax); c.dHi = c.smax + K_BOUND_RELAX * mx(1.0, c.smax);
    const double h[2] = {c.dtc, c.dt};
    for (int i = 0; i < 2; i++) {
        const double ld = c.sdmax * h[i], la = c.admax * h[i];
        double* dst = (i == 0) ? c.rHiFirst : c.rHiLater;
        dst[0] = ld + K_BOUND_RELAX * mx(1.0, ld);
        dst[1] = la + K_BOUND_RELAX * mx(1.0, la);
    }
    c.rfrac = c.Lb / (c.La + c.Lb);
    c.dtLb = c.dt / c.Lb;
    const double t = c.tol < 1e-4 ? c.tol : 1e-4;
    c.mu_min = t / (K_KAPPA_EPS + 1.0);
}

// ---- shared-memory layout of one warp, in doubles (every pair used by a 16-byte load is even-aligned) ----
#define W_P 0       // 6x6 cost-to-go Hessian, full symmetric storage, row stride 6
#define W_PV 36     // 6   cost-to-go gradient
#define W_TT 42     // 5x6: TT[c][i] = (P*M)[i][c] for c = psi,v,a,df and c = 4: P r + p
#define W_F 72      // 6x6 stage Hessian F over (x,y,psi,v,a,df)
#define W_FV 108    // 6   stage gradient f
#define W_EX 114    // 4(+2) unit vector e_x over rows (x,y,psi,v)
#define W_EY 120    // 4(+2) unit vector e_y
#define W_Z 126     // 6   zeros
#define W_C 132     // Ca, Cd of the current stage (copied from the record by idle lanes of round B)
#define W_NC 134    // (-Ca, 0), (0, -Cd) of the current stage
#define W_DUMMY 138 // sink for inactive lanes (2)
#define W_CONST 140 // problem constants: state[4], u_prev[2], v_des, pad
#define W_XCH 148   // teams of several warps only: exchange area (reductions, neighbour values, flags)
#define XCH_RED 0   //   [2][3][4] per-warp partial results of a reduction
#define XCH_DN 24   //   [2][3][8] first-lane values of each warp (read by the last lane of the warp below)
#define XCH_UP 72   //   [2][3][8] last-lane values of each warp (read by the first lane of the warp above)
#define XCH_FLAG 120 //  [2] broadcast scalars
#define XCH_SIZE 128
// stage records start at W_SD(W)
#define W_SD_OF(W) (148 + ((W) > 1 ? XCH_SIZE : 0))
// stage record
#define SD_CF 0     // 5 coefficient 4-vectors over next-state rows (x,y,psi,v): columns psi | v | a | df of [A B], then r
#define SD_R 16     //   r column (dynamics residual; record N: initial-condition residual)
#define SD_HXX 20
#define SD_HYY 21
#define SD_HPP 22
#define SD_HPV 23
#define SD_HVV 24
#define SD_HPD 25
#define SD_HVD 26
#define SD_HAA 27
#define SD_HDD 28
#define SD_CA 29
#define SD_CD 30
#define SD_ZERO 31  // constant 0 (H entries that are structurally zero point here)
#define SD_NCA 32   // -Ca
#define SD_NCD 33   // -Cd
#define SD_GX 34    // GX,GY,GP,GV,GA,GD (condensed gradient)
#define SD_SRW 40   // (Sigma_s + delta_w) of the rate row [steer, acc]
#define SD_BR 42    // -mu/ss_L + mu/ss_U of the rate row
#define SD_DR 44    // rate-row residual used as right-hand side
#define SDS 46      // even: records are 16-byte aligned
// Frenet-frame variant (MODEL 1, MKZMPCPathFollowerFrenet.jl): the stage map has dense s and e_y columns
// (rows s and e_psi depend on s through K(s) and on e_y) and a 5x5 Lagrangian-Hessian block over
// (s, e_y, e_psi, v, df).  Its record is the XY record (s, e_y, e_psi, v in the slots of x, y, psi, v) plus
#define SD_CS 46    // column s  of A over next-state rows (unit part included)
#define SD_CE 50    // column e_y of A
#define SD_HSE 54   // Hessian entries that are structurally zero in the XY model
#define SD_HSP 55
#define SD_HSV 56
#define SD_HSD 57
#define SD_HEP 58
#define SD_HEV 59
#define SD_HED 60
#define SDS_F 62
#define W_TT2 148   // MODEL 1: columns s | e_y of P M (2 x 6); the exchange area of multi-warp teams follows at 160
MPC_HD constexpr int sds_of(int model) { return model ? SDS_F : SDS; }
#define KST_STRIDE 14

// per-thread state kept in shared memory instead of registers, in groups: group g of stage k is the
// G_*_N doubles at  lf_offset(N) + G_*_OFF * (N + 2) + G_*_STRIDE * min(k, N + 1)   (slot N + 1 is shared
// by the threads that own no stage).  The strides are chosen so that 16-byte vector accesses of a
// quarter warp (8-byte ones of a half warp for REF) fall into distinct banks.
#define G_EV_OFF 0      // 12 (+2 pad): cos/sin(psi+beta), cos/sin(beta), beta', beta'', rd[4], dr[2] of the last evaluated point
#define G_EV_STRIDE 14
#define G_REF_OFF 14    // 3 (+1 so that the next group starts even): x_ref, y_ref, psi_ref
#define G_REF_STRIDE 3
#define G_DX_OFF 18     // 6: primal step dsx, dsy, dsp, dsv, dua, dud
#define G_DX_STRIDE 6
#define G_DRS_OFF 24    // 2: slack step of the rate row
#define G_DRS_STRIDE 2
#define G_DY_OFF 26     // 6: new equality / rate-row multipliers (y + dy)
#define G_DY_STRIDE 6
#define G_Z_OFF 32      // 10: bound multipliers zvL, zvU, zaL, zaU, zdL, zdU, rvL[2], rvU[2]
#define G_Z_STRIDE 10
#define LF_DOUBLES 42   // per stage slot, all groups
MPC_HD int team_warps(int N) { return (N + 1 + 31) / 32; }   // warps that share one problem
MPC_HD constexpr int w_sd_of(int W, int model) { return model ? 160 + (W > 1 ? XCH_SIZE : 0) : W_SD_OF(W); }   // MODEL 1: exchange area at 160
MPC_HD int lf_offset(int N, int model = 0) { return w_sd_of(team_warps(N), model) + (N + 1) * sds_of(model) + N * KST_STRIDE; }
MPC_HD int smem_doubles_per_team(int N, int model = 0, int pw = 0) { return lf_offset(N, model) + LF_DOUBLES * (N + 2) + (pw ? 8 : 0); }   // even: 16-byte alignment of the next team
// PW (per-problem weights) teams keep their problem's eight weights in update_cost order behind the rest of the team's area
MPC_HD int wt_offset(int N, int model) { return smem_doubles_per_team(N, model); }
// weight i (update_cost order of the XY model) of problem b in a caller's weight array: [B][8], or [B][7] for the Frenet-frame
// variant (cey, cep, cev, cda, cdd, ca, cd: the XY slots 1..7; nothing on s)
MPC_HD double row_weight(const double* w, long b, int i, int model) { return model ? (i ? w[7 * b + i - 1] : 0.0) : w[8 * b + i]; }
// the rule of mpcb200_set_cost: not negative and not NaN
MPC_HD bool row_weights_ok(const double* w, long b, int model) {
    bool ok = true;
    for (int i = 0; i < 8; i++) ok = ok && row_weight(w, b, i, model) >= 0.0;
    return ok;
}

MPC_DEV double dmax_(double a, double b) { return a > b ? a : b; }
MPC_DEV double dmin_(double a, double b) { return a < b ? a : b; }
MPC_DEV double warp_max(double v) {
    MPC_NOUNROLL for (int o = 16; o; o >>= 1) { double t = shfl_xor(v, o); v = (t > v || t != t) ? t : v; }
    return v;
}
MPC_DEV double warp_min(double v) {
    MPC_NOUNROLL for (int o = 16; o; o >>= 1) { double t = shfl_xor(v, o); v = (t < v) ? t : v; }
    return v;
}
MPC_DEV double warp_sum(double v) {
    MPC_NOUNROLL for (int o = 16; o; o >>= 1) v += shfl_xor(v, o);
    return v;
}
// inclusive suffix sum over lanes: out_k = sum_{j >= k} v_j
MPC_DEV double warp_suffix_sum(double v, int l) {
    MPC_NOUNROLL for (int o = 1; o < 32; o <<= 1) { double t = shfl_down(v, o); if (l + o < 32) v += t; }
    return v;
}
MPC_DEV void push_interior(double& v, double lo, double hi) {
    const double pl = dmin_(K_BOUND_PUSH * dmax_(1.0, fabs(lo)), K_BOUND_FRAC * (hi - lo));
    const double pu = dmin_(K_BOUND_PUSH * dmax_(1.0, fabs(hi)), K_BOUND_FRAC * (hi - lo));
    if (v < lo + pl) v = lo + pl;
    if (v > hi - pu) v = hi - pu;
}
MPC_DEV bool cmp_le(double lhs, double rhs, double bas) { return lhs - rhs <= 10.0 * K_EPS * fabs(bas); }

// The iterate: primal and equality multipliers stay in registers; the bound multipliers and the
// step live in per-thread shared-memory fields and are loaded by the routines that use them.
struct LaneState {
    double sx, sy, sp, sv, ua, ud;        // primal
    double yx, yy, yp, yv;                // multipliers of the equality rows that define s_k
    double rs[2], ryd[2];                 // rate row ending at u_k: slack, multiplier; [0] steering, [1] acceleration
};
struct BoundMult {
    double zvL, zvU, zaL, zaU, zdL, zdU;  // bound multipliers of v, acc, df
    double rvL[2], rvU[2];                // ... of the rate-row slacks
};
struct StepState {
    double dsx, dsy, dsp, dsv, dua, dud;  // primal step
    double drs[2];                        // slack step
    double nyx, nyy, nyp, nyv;            // NEW equality multipliers (y + dy)
    double nyd[2];                        // NEW rate-row multipliers
};
struct EvalLane {         // model evaluation at the last evaluated point, this thread's stage (lives in shared memory)
    double cs, sn, cb, sb, b1, b2;  // cos/sin(psi+beta), cos/sin(beta), beta', beta''
    double rd[4];         // k < N: f(s_k,u_k) - s_{k+1};  k = N: state - s_0;  else 0
    double dr[2];         // rate-row defect d(x) - slack
    double q, K;          // MODEL 1: 1 / (1 - e_y K(s)) and K(s)  (the two pad words of the group)
};
struct EvalState {        // ... and its team-wide scalars
    double f, lb, theta;  // objective (unscaled), sum of log slacks, 1-norm constraint violation
};
// reciprocals of the ten bound slacks of a lane, from ONE division
struct Recips { double vL, vU, aL, aU, dL, dU, r0L, r0U, r1L, r1U; };

struct Result { int status; int iters; double cost; int n_resto; };

// The two line-search tests that involve theta^s_theta / (-grad(phi)'d)^s_phi (Ipopt: FilterLSAcceptor::IsFtype and
// CalculateAlphaMin) are decided in double precision exactly as the oracle writes them; the single-precision
// estimate of the ratio only screens out the (almost all) cases that are more than 0.1 % away from the threshold.
//   form 0:  a (-gBd)^s_phi > delta theta^s_theta           form 1:  a > alpha_min_frac * delta theta^s_theta / (-gBd)^s_phi
MPC_DEV_NOINLINE bool ratio_test_exact(int form, double a, double theta, double mgbd) {
    if (form == 0) return a * pow(mgbd, K_S_PHI) > K_DELTA * pow(theta, K_S_THETA);
    return a > K_ALPHA_MIN_FRAC * (K_DELTA * pow(theta, K_S_THETA) / pow(mgbd, K_S_PHI));
}
MPC_DEV bool ratio_test(int form, double a, double thr32, double theta, double mgbd) {
    if (a > thr32 * 1.001) return true;
    if (a < thr32 * 0.999) return false;
    return ratio_test_exact(form, a, theta, mgbd);
}

// a / b for the rare branches: a call cannot be speculated, so the division (and its slow path for
// zero numerators) stays out of the common path
MPC_DEV_NOINLINE double div_cold(double a, double b) { return a / b; }

// kappa_sigma safeguard of the bound multipliers (Ipopt: correct_bound_multiplier); multipliers a
// thread does not own are 0 and stay 0.  Rare: out of line.
MPC_DEV_NOINLINE void kappa_sigma_clamp(double* z, const double* sl, double mu) {
    MPC_NOUNROLL for (int i = 0; i < 10; i++) {
        if (!(z[i] > 0.0)) continue;
        const double pz = z[i] * sl[i];
        if (pz > K_KAPPA_SIGMA * mu) z[i] = K_KAPPA_SIGMA * mu / sl[i];
        else if (pz * K_KAPPA_SIGMA < mu) z[i] = mu / (K_KAPPA_SIGMA * sl[i]);
    }
}

// Serial part of the restoration by rollout (see TeamSolver::rollout_restore): inputs of stage s are
// read from / written back to entries 4, 5 of stage s's step group, states written to entries 0..3.
// Rare (a few per cent of the cold starts, once each): out of line, scalars by value.
struct RolloutConsts { double dt, dtc, dtLb, rfrac, vmin, vmax, amax, smax, admax, sdmax; int model; double kp[4]; };
MPC_DEV_NOINLINE void rollout_core(smem_t sm, int fa, int cbase, int N, RolloutConsts c) {
    double s0 = lds(sm, cbase), s1 = lds(sm, cbase + SO(1)), s2 = lds(sm, cbase + SO(2)), s3 = lds(sm, cbase + SO(3));
    double pa = lds(sm, cbase + SO(5)), pd = lds(sm, cbase + SO(4));
    MPC_NOUNROLL for (int s = 0; s < N; s++) {
        double ua = lds(sm, fa + SO(4)), ud = lds(sm, fa + SO(5));
        if (s != 1) {   // rate rows exist for the first move and for pairs (s, s-1), s >= 2
            const double h = (s == 0) ? c.dtc : c.dt;
            const double la = 0.98 * c.admax * h, ld = 0.98 * c.sdmax * h;
            ua = dmin_(dmax_(ua, pa - la), pa + la);
            ud = dmin_(dmax_(ud, pd - ld), pd + ld);
        }
        ua = dmin_(dmax_(ua, -c.amax), c.amax);
        ud = dmin_(dmax_(ud, -c.smax), c.smax);
        ua = dmin_(dmax_(ua, (c.vmin - s3) / c.dt), (c.vmax - s3) / c.dt);   // v_{s+1} = v_s + dt acc stays inside [v_min, v_max]
        sts2(sm, fa, s0, s1); sts2(sm, fa + SO(2), s2, s3); sts2(sm, fa + SO(4), ua, ud);
        double sd, cd, sps, cps;
        mpc_sincos(ud, &sd, &cd);
        mpc_sincos(s2, &sps, &cps);
        const double r = c.rfrac;
        const double inv = sqrt(1.0 / (cd * cd + r * r * sd * sd));
        const double cb = cd * inv, sb = r * sd * inv;
        double n0 = s0 + c.dt * (s3 * (cps * cb - sps * sb));
        const double n1 = s1 + c.dt * (s3 * (sps * cb + cps * sb));
        double n2 = s2 + c.dtLb * (s3 * sb);
        const double n3 = s3 + c.dt * ua;
        if (c.model) {   // Frenet frame (MKZMPCPathFollowerFrenet.jl:111-120): (s, e_y, e_psi, v)
            const double K = ((c.kp[0] * s0 + c.kp[1]) * s0 + c.kp[2]) * s0 + c.kp[3];
            const double g = s3 * (cps * cb - sps * sb) / (1.0 - s1 * K);
            n0 = s0 + c.dt * g;
            n2 = s2 + (c.dtLb * (s3 * sb) - c.dt * (g * K));
        }
        s0 = n0; s1 = n1; s2 = n2; s3 = n3; pa = ua; pd = ud;
        fa += SO(G_DX_STRIDE);
    }
    sts2(sm, fa, s0, s1); sts2(sm, fa + SO(2), s2, s3); sts2(sm, fa + SO(4), 0.0, 0.0);
}

// ---- lane roles of the Riccati backward recursion (lanes = matrix entries), one row of ROLE_STRIDE
// ints per lane: shared-memory offsets (SO units) of the operands of rounds A, B and E.  They depend
// only on the lane, the horizon and the team size, so mpcb200_create computes the table once.
#define ROLE_STRIDE 20
#define ROLE_STRIDE_F 24   // MODEL 1: + second task of round A (columns s | e_y of P M, lanes 0..11): a2_p, a2_m, a2_out
MPC_HD constexpr int role_stride_of(int model) { return model ? ROLE_STRIDE_F : ROLE_STRIDE; }
MPC_HD void riccati_roles(int l, int N, int W_SD, int* out, int model = 0) {
    const int SDS_ = sds_of(model);
    int a_p, a_m, a_ex, a_out, b_m, b_mk, b_t, b_x, b_h, b_o1, b_o2, e_f0, e_fi, e_fj, e_o1, e_o2, e_k0, e_k1;
        {
            // round A: lane (i, cc) -> TT[cc][i] = sum_{j<4} P[i][j] CF[cc][j] + X,  X = 0 | P[i][4] | P[i][5] | p[i]
            const int i = (l < 24) ? (l >> 2) : (l < 30 ? l - 24 : 0);
            const int cc = (l < 24) ? (l & 3) : 4;
            a_p = (SO(W_P + 6 * i));
            a_m = (SO(W_SD + SD_CF + 4 * cc));
            a_ex = ((l >= 30) ? SO(W_Z) : (cc == 2) ? SO(W_P + 6 * i + 4) : (cc == 3) ? SO(W_P + 6 * i + 5) : (cc == 4) ? SO(W_PV + i) : SO(W_Z));
            a_out = ((l < 30) ? SO(W_TT + 6 * cc + i) : SO(W_DUMMY));
        }
        {
            // round B: 21 symmetric pairs (c1 <= c2) over (x,y,psi,v,a,df); 6 vector entries; 4 copy lanes
            //   F[c1][c2] = H + sum_{i<4} M[i][c1] That[i][c2] + X,  X = That[4][c2] (c1 = a) | That[5][c2] (c1 = df) | 0
            int c1 = 0, c2 = 0, kind = 0;  // 0 pair, 1 vector, 2 copy, 3 idle
            if (l < 21) { int t = l; while (t >= 6 - c1) { t -= 6 - c1; c1++; } c2 = c1 + t; }
            else if (l < 27) { c1 = l - 21; kind = 1; }
            else if (l < 31) kind = 2;
            else kind = 3;
            int mb, mk, tb, xb, hf, o1, o2;
            if (kind >= 2) { mb = SO(W_Z); mk = 0; }
            else if (c1 < 2 && model) { mb = SO(W_SD + (c1 == 0 ? SD_CS : SD_CE)); mk = 1; }
            else if (c1 < 2) { mb = (c1 == 0) ? SO(W_EX) : SO(W_EY); mk = 0; }
            else { mb = SO(W_SD + SD_CF + 4 * (c1 - 2)); mk = 1; }
            // That column c2 (rows 0..5 contiguous): P row c2 (symmetric) for x,y; TT column otherwise; TT[4] for the vector
            if (kind == 1) tb = SO(W_TT + 24);
            else if (kind == 0) tb = (c2 < 2) ? (model ? SO(W_TT2 + 6 * c2) : SO(W_P + 6 * c2)) : SO(W_TT + 6 * (c2 - 2));
            else tb = SO(W_Z);
            xb = (kind <= 1 && c1 == 4) ? tb + SO(4) : (kind <= 1 && c1 == 5) ? tb + SO(5) : SO(W_Z);
            hf = SD_ZERO;
            if (kind == 1) hf = SD_GX + c1;
            else if (kind == 0) {
                if (c1 == c2) hf = (c1 == 0) ? SD_HXX : (c1 == 1) ? SD_HYY : (c1 == 2) ? SD_HPP : (c1 == 3) ? SD_HVV : (c1 == 4) ? SD_HAA : SD_HDD;
                else if (c1 == 2 && c2 == 3) hf = SD_HPV;
                else if (c1 == 2 && c2 == 5) hf = SD_HPD;
                else if (c1 == 3 && c2 == 5) hf = SD_HVD;
                else if (model && c1 == 0 && c2 == 1) hf = SD_HSE;
                else if (model && c1 == 0 && c2 == 2) hf = SD_HSP;
                else if (model && c1 == 0 && c2 == 3) hf = SD_HSV;
                else if (model && c1 == 0 && c2 == 5) hf = SD_HSD;
                else if (model && c1 == 1 && c2 == 2) hf = SD_HEP;
                else if (model && c1 == 1 && c2 == 3) hf = SD_HEV;
                else if (model && c1 == 1 && c2 == 5) hf = SD_HED;
            } else if (kind == 2) hf = (l == 27) ? SD_CA : (l == 28) ? SD_CD : (l == 29) ? SD_NCA : SD_NCD;
            if (kind == 0) { o1 = SO(W_F + 6 * c1 + c2); o2 = SO(W_F + 6 * c2 + c1); }
            else if (kind == 1) { o1 = o2 = SO(W_FV + c1); }
            else if (kind == 2) { o1 = o2 = (l == 27) ? SO(W_C) : (l == 28) ? SO(W_C + 1) : (l == 29) ? SO(W_NC) : SO(W_NC + 3); }
            else { o1 = o2 = SO(W_DUMMY); }
            b_m = (mb); b_mk = (mk); b_t = (tb); b_x = (xb); b_h = (SO(W_SD + hf));
            b_o1 = (o1); b_o2 = (o2);
        }
        {
            // 21 symmetric pairs (i <= j) over xi, then 6 vector entries.
            // P'[i][j] = F8[i][j] + F8[i][a] K[0][j] + F8[i][df] K[1][j],  K[.][j] = -Fuu^{-1} (F8[j][a], F8[j][df])
            int i = 0, j = 0, vec = 0, act = 1;
            if (l < 21) { int t = l; while (t >= 6 - i) { t -= 6 - i; i++; } j = i + t; }
            else if (l < 27) { i = l - 21; vec = 1; }
            else act = 0;
            int f0;
            if (vec) f0 = (i < 4) ? SO(W_FV + i) : SO(W_Z);
            else if (i < 4 && j < 4) f0 = SO(W_F + 6 * i + j);
            else if (i == 4 && j == 4) f0 = SO(W_C);
            else if (i == 5 && j == 5) f0 = SO(W_C + 1);
            else f0 = SO(W_Z);
            auto pairof = [](int q) {   // (F8[q][a], F8[q][df]) for q over xi; q = 6: (f_a, f_df)
                return (q < 4) ? SO(W_F + 6 * q + 4) : (q == 4) ? SO(W_NC) : (q == 5) ? SO(W_NC + 2) : SO(W_FV + 4);
            };
            const int fi = pairof(i), fj = pairof(vec ? 6 : j);
            int o1, o2;
            if (!act) { o1 = o2 = SO(W_DUMMY); }
            else if (vec) { o1 = o2 = SO(W_PV + i); }
            else { o1 = SO(W_P + 6 * i + j); o2 = SO(W_P + 6 * j + i); }
            // gain storage: the diagonal pairs (j,j) hold K[.][j], vector lane i = 0 holds K[.][6]
            int ks = -1;
            if (act && !vec && i == j) ks = j;
            if (act && vec && i == 0) ks = 6;
            const int kb = SO(W_SD + (N + 1) * SDS_ + (N - 1) * KST_STRIDE);  // gains of stage N-1
            e_f0 = (f0); e_fi = (fi); e_fj = (fj); e_o1 = (o1); e_o2 = (o2);
            e_k0 = (ks >= 0 ? kb + SO(ks) : SO(W_DUMMY));
            e_k1 = (ks >= 0 ? kb + SO(7 + ks) : SO(W_DUMMY));
        }
    out[0] = a_p; out[1] = a_m; out[2] = a_ex; out[3] = a_out; out[4] = b_m; out[5] = b_mk; out[6] = b_t; out[7] = b_x; out[8] = b_h;
    out[9] = b_o1; out[10] = b_o2; out[11] = e_f0; out[12] = e_fi; out[13] = e_fj; out[14] = e_o1; out[15] = e_o2;
    out[16] = e_k0; out[17] = e_k1; out[18] = (e_k0 == SO(W_DUMMY)) ? 0 : SO(KST_STRIDE); out[19] = 0;
    if (model) {
        // second task of round A: lane (i, cc) for l < 12 -> TT2[cc][i] = sum_{j<4} P[i][j] C[cc][j], C = column s | e_y of A
        const int i = (l < 12) ? (l >> 1) : 0, cc = l & 1;
        out[20] = SO(W_P + 6 * i);
        out[21] = (l < 12) ? SO(W_SD + (cc ? SD_CE : SD_CS)) : SO(W_SD + SD_CS);
        out[22] = (l < 12) ? SO(W_TT2 + 6 * cc + i) : SO(W_DUMMY);
        out[23] = 0;
    }
}

// ---- reference generation on the device (scripts/gps_utils/ref_gps_traj.py:131-218), used by the
// closed-loop rollout and by mpcb200_solve_batch_on_path (TeamSolver::get_waypoints)
struct PathTable {
    const double *t, *X, *Y, *psi, *s; int n;   // columns 0,4,5,3,6 of ref_gps_traj.py:106
    const double* cb; int nch;                  // bounding circles of chunks of PATH_CHUNK samples: cx[nch], cy[nch], r[nch] (null: none)
};
#define PATH_CHUNK 16
inline int path_chunks(int n) { return (n + PATH_CHUNK - 1) / PATH_CHUNK; }
// host: the bounding circles for nearest_sample: centre of the chunk's bounding box, radius = largest distance to one of its
// samples, inflated so that rounding can only make a circle larger than the samples need
inline void path_chunk_bounds(int n, const double* X, const double* Y, double* out) {
    const int nch = path_chunks(n);
    for (int c = 0; c < nch; c++) {
        const int i0 = c * PATH_CHUNK, i1 = (i0 + PATH_CHUNK < n) ? i0 + PATH_CHUNK : n;
        double x0 = X[i0], x1 = X[i0], y0 = Y[i0], y1 = Y[i0];
        for (int i = i0; i < i1; i++) { x0 = X[i] < x0 ? X[i] : x0; x1 = X[i] > x1 ? X[i] : x1; y0 = Y[i] < y0 ? Y[i] : y0; y1 = Y[i] > y1 ? Y[i] : y1; }
        const double cx = 0.5 * (x0 + x1), cy = 0.5 * (y0 + y1);
        double r2 = 0.0;
        for (int i = i0; i < i1; i++) { const double dx = X[i] - cx, dy = Y[i] - cy, d = dx * dx + dy * dy; r2 = d > r2 ? d : r2; }
        out[c] = cx; out[nch + c] = cy;
        out[2 * nch + c] = sqrt(r2) * (1.0 + 1e-9) + 1e-12 * (fabs(cx) + fabs(cy)) + 1e-300;
    }
}

// np.interp(xq, xp, fp): every operation rounded on its own like numpy's compiled loop (no FMA contraction)
MPC_DEV double np_interp(double xq, const double* xp, const double* fp, int n) {
    if (xq <= xp[0]) return fp[0];
    if (xq >= xp[n - 1]) return fp[n - 1];
    int lo = 0, hi = n - 1;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (xp[mid] <= xq) lo = mid; else hi = mid; }
    const double slope = (fp[lo + 1] - fp[lo]) / (xp[lo + 1] - xp[lo]);
    return add_rn(mul_rn(slope, xq - xp[lo]), fp[lo]);
}

// ---- lane roles of the REGISTER version of the Riccati backward recursion (MODEL 0): the cost-to-go P (one entry per
// lane), the products P M and the stage Hessian F never leave registers; operands move between lanes with warp shuffles.
// Per lane: source lanes of the shuffles of rounds A, B and E (five 5-bit fields per int), shared-memory offsets of the
// operands that still come from the stage record, and a few flags.
#define RS_STRIDE 12
//   [0] A: source lanes of P[i][0..3] and of the extra term, 5 bits each      [1] A: offset of column cc of [A B] in the record
//   [2] B: source lanes of That[0..3][c2] and of the extra term                [3] B: offset of column c1 of M (record or constant area)
//   [4] B: 1 if that offset is relative to the current record                  [5] B: offset of the H / g entry in the record
//   [6] E: source lanes of F[i][a], F[i][df], F[j][a], F[j][df]                [7] flags (RSF_*)
//   [8], [9] gain addresses of stage N-1 (or the sink)   [10] gain step per stage   [11] pad
#define RSF_B_OWN 2      // round B: F = H + own P entry (both columns are unit vectors)
// Lane 31 holds 0 in all three registers at all times (its operands are zeros), so "no extra term" is a shuffle from
// lane 31; in round B the otherwise idle lanes 27..30 pick up -Ca, -Cd, Ca, Cd from the record, which round E reads for the
// rows a_prev / df_prev of F8 -- no selects in the loop except RSF_B_OWN.
#define RS_ZERO_LANE 31
#define RS_NCA_LANE 27
#define RS_NCD_LANE 28
#define RS_CA_LANE 29
#define RS_CD_LANE 30
MPC_HD int pair_lane(int i, int j) { if (i > j) { const int t = i; i = j; j = t; } return i * 6 - i * (i - 1) / 2 + (j - i); }
MPC_HD void riccati_roles_shfl(int l, int N, int W_SD, int* out) {
    int flags = 0;
    const int Z = RS_ZERO_LANE;
    {   // round A: lane (i, cc) -> TT[cc][i] = sum_{j<4} P[i][j] CF[cc][j] + X,  X = 0 | P[i][4] | P[i][5] | p[i]
        const int i = (l < 24) ? (l >> 2) : (l < 30 ? l - 24 : 0);
        const int cc = (l < 24) ? (l & 3) : 4;
        int src = 0, sx = Z;
        for (int j = 0; j < 4; j++) src |= ((l < 30) ? pair_lane(i, j) : Z) << (5 * j);
        if (l < 30 && cc == 2) sx = pair_lane(i, 4);
        if (l < 30 && cc == 3) sx = pair_lane(i, 5);
        if (l < 30 && cc == 4) sx = 21 + i;
        out[0] = src | (sx << 20);
        out[1] = (l < 30) ? SO(W_SD + SD_CF + 4 * cc) : SO(W_Z);
        out[11] = (l < 30) ? 1 : 0;    // offset relative to the current record
    }
    {   // round B: 21 symmetric pairs (c1 <= c2) over (x,y,psi,v,a,df); 6 vector entries; lanes 27..30 stage -Ca, -Cd, Ca, Cd
        int c1 = 0, c2 = 0, kind = 0;  // 0 pair, 1 vector, 3 other
        if (l < 21) { int t = l; while (t >= 6 - c1) { t -= 6 - c1; c1++; } c2 = c1 + t; }
        else if (l < 27) { c1 = l - 21; kind = 1; }
        else kind = 3;
        int src = Z | (Z << 5) | (Z << 10) | (Z << 15), sx = Z, mb = SO(W_Z), mk = 0, hf = SD_ZERO;
        if (kind == 0 && c2 < 2) flags |= RSF_B_OWN;
        if (kind <= 1) {
            const int col = (kind == 1) ? 4 : (c2 >= 2 ? c2 - 2 : 0);              // TT column that is That[.][c2]
            src = 0;
            for (int r = 0; r < 4; r++) src |= ((col == 4) ? 24 + r : 4 * r + col) << (5 * r);
            if (c1 >= 4) sx = (col == 4) ? 24 + c1 : 4 * c1 + col;
            if (c1 < 2) { mb = (c1 == 0) ? SO(W_EX) : SO(W_EY); mk = 0; }
            else { mb = SO(W_SD + SD_CF + 4 * (c1 - 2)); mk = 1; }
            if (kind == 1) hf = SD_GX + c1;
            else if (c1 == c2) hf = (c1 == 0) ? SD_HXX : (c1 == 1) ? SD_HYY : (c1 == 2) ? SD_HPP : (c1 == 3) ? SD_HVV : (c1 == 4) ? SD_HAA : SD_HDD;
            else if (c1 == 2 && c2 == 3) hf = SD_HPV;
            else if (c1 == 2 && c2 == 5) hf = SD_HPD;
            else if (c1 == 3 && c2 == 5) hf = SD_HVD;
        } else {
            hf = (l == RS_NCA_LANE) ? SD_NCA : (l == RS_NCD_LANE) ? SD_NCD : (l == RS_CA_LANE) ? SD_CA : (l == RS_CD_LANE) ? SD_CD : SD_ZERO;
        }
        out[2] = src | (sx << 20); out[3] = mb; out[4] = mk; out[5] = SO(W_SD + hf);
    }
    {   // round E: 21 symmetric pairs (i <= j) over xi = (x,y,psi,v,a_prev,df_prev), then 6 vector entries
        int i = 0, j = 0, vec = 0, act = 1;
        if (l < 21) { int t = l; while (t >= 6 - i) { t -= 6 - i; i++; } j = i + t; }
        else if (l < 27) { i = l - 21; vec = 1; }
        else act = 0;
        // (F8[q][a], F8[q][df]) for q over xi; q = 6: (f_a, f_df)
        int six = Z, siy = Z, sjx = Z, sjy = Z, sf0 = Z;
        if (act) {
            if (i < 4) { six = pair_lane(i, 4); siy = pair_lane(i, 5); }
            else if (i == 4) six = RS_NCA_LANE;
            else siy = RS_NCD_LANE;
            const int q = vec ? 6 : j;
            if (q < 4) { sjx = pair_lane(q, 4); sjy = pair_lane(q, 5); }
            else if (q == 4) sjx = RS_NCA_LANE;
            else if (q == 5) sjy = RS_NCD_LANE;
            else { sjx = 21 + 4; sjy = 21 + 5; }
            if (vec) sf0 = (i < 4) ? l : Z;
            else if (i < 4 && j < 4) sf0 = l;
            else if (i == 4 && j == 4) sf0 = RS_CA_LANE;
            else if (i == 5 && j == 5) sf0 = RS_CD_LANE;
        }
        out[6] = six | (siy << 5) | (sjx << 10) | (sjy << 15) | (sf0 << 20);
        int ks = -1;   // gain storage: the diagonal pairs (j,j) hold K[.][j], vector lane i = 0 holds K[.][6]
        if (act && !vec && i == j) ks = j;
        if (act && vec && i == 0) ks = 6;
        const int kb = SO(W_SD + (N + 1) * SDS + (N - 1) * KST_STRIDE);  // gains of stage N-1
        out[8] = (ks >= 0 ? kb + SO(ks) : SO(W_DUMMY));
        out[9] = (ks >= 0 ? kb + SO(7 + ks) : SO(W_DUMMY));
        out[10] = (ks >= 0) ? SO(KST_STRIDE) : 0;
    }
    out[7] = flags;
}

// W = warps per team (1: a warp per problem; 2, 3: a block per problem)
// MODEL 0: XY kinematic bicycle (MKZMPCPathFollower.jl); MODEL 1: Frenet-frame variant (MKZMPCPathFollowerFrenet.jl)
// PW: the cost weights are this problem's (wt_offset in the team's shared memory, staged by solve_problem / rollout_group) instead
// of the kernel parameter KCfg::w.  PW = 0 reads the kernel parameter, as the unweighted entry points always have.
template <int W, int MODEL = 0, int PW = 0>
struct TeamSolver {
    static constexpr int W_XCHG = MODEL ? 160 : W_XCH;   // exchange area of multi-warp teams
    static constexpr int W_SD = w_sd_of(W, MODEL);   // first stage record
    static constexpr int SDSZ = sds_of(MODEL);       // doubles per stage record
    static constexpr int NFILT_MAX = 32 * W;  // one filter entry per thread
    const KCfg& c;
    const smem_t sm;   // this team's shared memory (opaque base)
    const int k;       // thread of the team = stage
    const int N;
    const bool isS, isU, isR;  // thread owns a state / an input / a rate row
    int xpar;                  // W > 1: parity of the exchange buffers
    const int slot;            // this thread's slot in the per-thread state groups: min(k, N + 1)
    double sigma;
    LaneState L;
    EvalState ev;

    MPC_DEV static int team_tid() { return (W == 1) ? lane_id() : thread_in_block(); }
    MPC_DEV TeamSolver(const KCfg& cfg, smem_t smem)
        : c(cfg), sm(smem), k(team_tid()), N(cfg.N), isS(team_tid() <= cfg.N), isU(team_tid() < cfg.N),
          isR((team_tid() == 0 || team_tid() >= 2) && team_tid() < cfg.N), xpar(0),
          slot(team_tid() <= cfg.N ? team_tid() : cfg.N + 1) {}

    // per-thread state in shared memory (groups G_*)
    MPC_DEV int grp(int off, int stride) const { return SO(lf_offset(N, MODEL) + off * (N + 2)) + slot * SO(stride); }
    MPC_DEV void ev_store(const EvalLane& e) {
        const int a = grp(G_EV_OFF, G_EV_STRIDE);
        sts2(sm, a, e.cs, e.sn); sts2(sm, a + SO(2), e.cb, e.sb); sts2(sm, a + SO(4), e.b1, e.b2);
        sts2(sm, a + SO(6), e.rd[0], e.rd[1]); sts2(sm, a + SO(8), e.rd[2], e.rd[3]); sts2(sm, a + SO(10), e.dr[0], e.dr[1]);
        if (MODEL) sts2(sm, a + SO(12), e.q, e.K);
    }
    MPC_DEV void ev_load_model(EvalLane& e) const {
        const int a = grp(G_EV_OFF, G_EV_STRIDE);
        const d2 v0 = lds2(sm, a), v1 = lds2(sm, a + SO(2)), v2 = lds2(sm, a + SO(4));
        e.cs = v0.x; e.sn = v0.y; e.cb = v1.x; e.sb = v1.y; e.b1 = v2.x; e.b2 = v2.y;
        if (MODEL) { const d2 v3 = lds2(sm, a + SO(12)); e.q = v3.x; e.K = v3.y; }
    }
    MPC_DEV void ev_load_resid(EvalLane& e) const {
        const int a = grp(G_EV_OFF, G_EV_STRIDE);
        const d2 v0 = lds2(sm, a + SO(6)), v1 = lds2(sm, a + SO(8)), v2 = lds2(sm, a + SO(10));
        e.rd[0] = v0.x; e.rd[1] = v0.y; e.rd[2] = v1.x; e.rd[3] = v1.y; e.dr[0] = v2.x; e.dr[1] = v2.y;
    }
    MPC_DEV void set_ref(double x, double y, double p) {
        const int a = grp(G_REF_OFF, G_REF_STRIDE);
        sts(sm, a, x); sts(sm, a + SO(1), y); sts(sm, a + SO(2), p);
    }
    // MODEL 1: the cost is on e_y, e_psi themselves (reference 0); the reference group holds each thread's copy of
    // the curvature polynomial instead (4 doubles, the group's full width)
    MPC_DEV double ref_x() const { return MODEL ? 0.0 : lds(sm, grp(G_REF_OFF, G_REF_STRIDE)); }
    MPC_DEV double ref_y() const { return MODEL ? 0.0 : lds(sm, grp(G_REF_OFF, G_REF_STRIDE) + SO(1)); }
    MPC_DEV double ref_p() const { return MODEL ? 0.0 : lds(sm, grp(G_REF_OFF, G_REF_STRIDE) + SO(2)); }
    MPC_DEV void set_kpoly(double k0, double k1, double k2, double k3) {
        const int a = grp(G_REF_OFF, 4);
        sts2(sm, a, k0, k1); sts2(sm, a + SO(2), k2, k3);
    }
    // curvature K(s) and its derivatives at this thread's s (MKZMPCPathFollowerFrenet.jl:111)
    struct Curv { double K, K1, K2; };
    MPC_DEV Curv curvature(double s) const {
        const int a = grp(G_REF_OFF, 4);
        const d2 k01 = lds2(sm, a), k23 = lds2(sm, a + SO(2));
        Curv r;
        r.K = ((k01.x * s + k01.y) * s + k23.x) * s + k23.y;
        r.K1 = (3.0 * k01.x * s + 2.0 * k01.y) * s + k23.x;
        r.K2 = 6.0 * k01.x * s + 2.0 * k01.y;
        return r;
    }
    MPC_DEV void ld_dx(StepState& D) const {
        const int a = grp(G_DX_OFF, G_DX_STRIDE);
        const d2 v0 = lds2(sm, a), v1 = lds2(sm, a + SO(2)), v2 = lds2(sm, a + SO(4));
        D.dsx = v0.x; D.dsy = v0.y; D.dsp = v1.x; D.dsv = v1.y; D.dua = v2.x; D.dud = v2.y;
    }
    MPC_DEV void st_dx(const StepState& D) {
        const int a = grp(G_DX_OFF, G_DX_STRIDE);
        sts2(sm, a, D.dsx, D.dsy); sts2(sm, a + SO(2), D.dsp, D.dsv); sts2(sm, a + SO(4), D.dua, D.dud);
    }
    MPC_DEV void ld_drs(StepState& D) const { const d2 v = lds2(sm, grp(G_DRS_OFF, G_DRS_STRIDE)); D.drs[0] = v.x; D.drs[1] = v.y; }
    MPC_DEV void st_drs(const StepState& D) { sts2(sm, grp(G_DRS_OFF, G_DRS_STRIDE), D.drs[0], D.drs[1]); }
    MPC_DEV void ld_dy(StepState& D) const {
        const int a = grp(G_DY_OFF, G_DY_STRIDE);
        const d2 v0 = lds2(sm, a), v1 = lds2(sm, a + SO(2)), v2 = lds2(sm, a + SO(4));
        D.nyx = v0.x; D.nyy = v0.y; D.nyp = v1.x; D.nyv = v1.y; D.nyd[0] = v2.x; D.nyd[1] = v2.y;
    }
    MPC_DEV void st_dy(const StepState& D) {
        const int a = grp(G_DY_OFF, G_DY_STRIDE);
        sts2(sm, a, D.nyx, D.nyy); sts2(sm, a + SO(2), D.nyp, D.nyv); sts2(sm, a + SO(4), D.nyd[0], D.nyd[1]);
    }
    MPC_DEV void ld_z(BoundMult& Z) const {
        const int a = grp(G_Z_OFF, G_Z_STRIDE);
        const d2 v0 = lds2(sm, a), v1 = lds2(sm, a + SO(2)), v2 = lds2(sm, a + SO(4)), v3 = lds2(sm, a + SO(6)), v4 = lds2(sm, a + SO(8));
        Z.zvL = v0.x; Z.zvU = v0.y; Z.zaL = v1.x; Z.zaU = v1.y; Z.zdL = v2.x; Z.zdU = v2.y;
        Z.rvL[0] = v3.x; Z.rvL[1] = v3.y; Z.rvU[0] = v4.x; Z.rvU[1] = v4.y;
    }
    MPC_DEV void st_z(const BoundMult& Z) {
        const int a = grp(G_Z_OFF, G_Z_STRIDE);
        sts2(sm, a, Z.zvL, Z.zvU); sts2(sm, a + SO(2), Z.zaL, Z.zaU); sts2(sm, a + SO(4), Z.zdL, Z.zdU);
        sts2(sm, a + SO(6), Z.rvL[0], Z.rvL[1]); sts2(sm, a + SO(8), Z.rvU[0], Z.rvU[1]);
    }

    // ------------------------------------------------------------------
    // team collectives.  W == 1: plain warp shuffles.  W > 1: warp shuffles, then the values that
    // cross a warp boundary go through the exchange area (double-buffered by `xpar`, so that one
    // bar.sync per collective suffices).
    // ------------------------------------------------------------------
    MPC_DEV void tsync() { if (W == 1) syncwarp(); else block_sync(); }
    MPC_DEV bool tall(bool p) { if (W == 1) return warp_all(p); else return block_all(p); }
    MPC_DEV int xflip() { const int b = xpar; xpar ^= 1; return b; }
    enum { OP_SUM = 0, OP_MAX = 1, OP_MIN = 2 };
    template <int OP> MPC_DEV static double comb(double a, double b) {
        if (OP == OP_SUM) return a + b;
        if (OP == OP_MAX) return (b > a || b != b) ? b : a;   // NaN wins, like warp_max
        return (b < a) ? b : a;
    }
    // all-reduce of n (<= 3) values at once (interleaved butterflies)
    template <int OP, int n> MPC_DEV void treduce(double* v) {
        MPC_NOUNROLL for (int o = 16; o; o >>= 1) {
            double t[n];
            for (int j = 0; j < n; j++) t[j] = shfl_xor(v[j], o);
            for (int j = 0; j < n; j++) v[j] = comb<OP>(v[j], t[j]);
        }
        if (W > 1) {
            const int base = SO(W_XCHG + XCH_RED + xflip() * 12);
            if (lane_id() == 0) for (int j = 0; j < n; j++) sts(sm, base + SO((k >> 5) * 4 + j), v[j]);
            block_sync();
            for (int j = 0; j < n; j++) {
                double a = lds(sm, base + SO(j));
                for (int w = 1; w < W; w++) a = comb<OP>(a, lds(sm, base + SO(w * 4 + j)));
                v[j] = a;
            }
        }
    }
    MPC_DEV double tsum(double v) { treduce<OP_SUM, 1>(&v); return v; }
    MPC_DEV double tmax(double v) { treduce<OP_MAX, 1>(&v); return v; }
    MPC_DEV double tmin(double v) { treduce<OP_MIN, 1>(&v); return v; }
    // inclusive suffix sums over stages of n (<= 2) values at once: out_k = sum_{j >= k} v_j
    template <int n> MPC_DEV void tsuffix(double* v) {
        const int l = lane_id();
        MPC_NOUNROLL for (int o = 1; o < 32; o <<= 1) {
            double t[n];
            for (int j = 0; j < n; j++) t[j] = shfl_down(v[j], o);
            if (l + o < 32) for (int j = 0; j < n; j++) v[j] += t[j];
        }
        if (W > 1) {
            const int base = SO(W_XCHG + XCH_RED + xflip() * 12);
            if (l == 0) for (int j = 0; j < n; j++) sts(sm, base + SO((k >> 5) * 4 + j), v[j]);   // this warp's total
            block_sync();
            for (int w = W - 1; w > (k >> 5); w--) for (int j = 0; j < n; j++) v[j] += lds(sm, base + SO(w * 4 + j));
        }
    }
    // neighbour exchange of nd values downwards (out = value of stage k+1) and nu values upwards
    // (out = value of stage k-1) in one step.  wrapN >= 0: thread wrapN receives stage 0's `dn` values.
    // Threads without that neighbour get an unspecified finite value.
    template <int nd, int nu, bool WRAP> MPC_DEV void xchg(const double* dn, double* dn_out, const double* up, double* up_out, int wrapN = -1) {
        if (W == 1) {
            const int src = (k == wrapN) ? 0 : ((k + 1) & 31);
            for (int j = 0; j < nd; j++) dn_out[j] = WRAP ? shfl(dn[j], src) : shfl_down(dn[j], 1);
            for (int j = 0; j < nu; j++) up_out[j] = shfl_up(up[j], 1);
        } else {
            const int l = lane_id(), w = k >> 5;
            for (int j = 0; j < nd; j++) dn_out[j] = shfl_down(dn[j], 1);
            for (int j = 0; j < nu; j++) up_out[j] = shfl_up(up[j], 1);
            const int b = xflip();
            const int bd = SO(W_XCHG + XCH_DN + b * 24), bu = SO(W_XCHG + XCH_UP + b * 24);
            if (l == 0) for (int j = 0; j < nd; j++) sts(sm, bd + SO(w * 8 + j), dn[j]);
            if (l == 31) for (int j = 0; j < nu; j++) sts(sm, bu + SO(w * 8 + j), up[j]);
            block_sync();
            if (l == 31 && w + 1 < W) for (int j = 0; j < nd; j++) dn_out[j] = lds(sm, bd + SO((w + 1) * 8 + j));
            if (l == 0 && w > 0) for (int j = 0; j < nu; j++) up_out[j] = lds(sm, bu + SO((w - 1) * 8 + j));
            if (WRAP && k == wrapN) for (int j = 0; j < nd; j++) dn_out[j] = lds(sm, bd + SO(j));
        }
    }
    template <int n> MPC_DEV void xnext(const double* in, double* out) { xchg<n, 0, false>(in, out, nullptr, nullptr); }
    template <int n> MPC_DEV void xprev(const double* in, double* out) { xchg<0, n, false>(nullptr, nullptr, in, out); }
    // value held by stage 0, for every thread
    MPC_DEV double bcast0(double v) {
        if (W == 1) return shfl(v, 0);
        const int a = SO(W_XCHG + XCH_FLAG + xflip());
        if (k == 0) sts(sm, a, v);
        block_sync();
        return lds(sm, a);
    }

    // value held by stage `src`, for every thread
    MPC_DEV double bcast_from(double v, int src) {
        if (W == 1) return shfl(v, src);
        const int a = SO(W_XCHG + XCH_FLAG + xflip());
        if (k == src) sts(sm, a, v);
        block_sync();
        return lds(sm, a);
    }
    // smallest (d, i) pair over the team, ties to the smaller index (numpy argmin returns the first minimum)
    MPC_DEV void targmin(double& d, int& i) {
        MPC_NOUNROLL for (int o = 16; o; o >>= 1) {
            const double od = shfl_xor(d, o); const int oi = shfl(i, lane_id() ^ o);
            if (od < d || (od == d && oi < i)) { d = od; i = oi; }
        }
        if (W > 1) {
            const int base = SO(W_XCHG + XCH_RED + xflip() * 12);
            if (lane_id() == 0) { sts(sm, base + SO((k >> 5) * 4), d); sts(sm, base + SO((k >> 5) * 4 + 1), (double)i); }
            block_sync();
            d = lds(sm, base); i = (int)lds(sm, base + SO(1));
            for (int w = 1; w < W; w++) {
                const double od = lds(sm, base + SO(w * 4)); const int oi = (int)lds(sm, base + SO(w * 4 + 1));
                if (od < d || (od == d && oi < i)) { d = od; i = oi; }
            }
        }
    }

    // cheap per-use reconstruction of lane constants (keeps them out of the register file)
    MPC_DEV double wt(int i) const { return PW ? lds(sm, SO(wt_offset(N, MODEL) + i)) : c.w[i]; }   // cost weight i (update_cost order)
    MPC_DEV double wx() const { return (k >= 1 && k <= N) ? wt(0) : 0.0; }
    MPC_DEV double wy() const { return (k >= 1 && k <= N) ? wt(1) : 0.0; }
    MPC_DEV double wp() const { return (k >= 1 && k <= N) ? wt(2) : 0.0; }
    MPC_DEV double wv() const { return (k >= 1 && k <= N - 1) ? wt(3) : 0.0; }
    MPC_DEV double rHi(int i) const { return (k == 0) ? c.rHiFirst[i] : c.rHiLater[i]; }
    MPC_DEV double cst(int i) const { return lds(sm, SO(W_CONST + i)); }  // state[0..3], u_prev[0..1], v_des
    MPC_DEV int rec() const { return SO(W_SD + (isS ? k : 0) * SDSZ); }    // this lane's own stage record

    MPC_DEV static void init_work(smem_t sm, int N) {
        const int l = team_tid();
        if (l < 6) { sts(sm, SO(W_EX + l), (l == 0) ? 1.0 : 0.0); sts(sm, SO(W_EY + l), (l == 1) ? 1.0 : 0.0); sts(sm, SO(W_Z + l), 0.0); }
        if (l < 4) sts(sm, SO(W_NC + l), 0.0);
        if (l < 2) sts(sm, SO(W_DUMMY + l), 0.0);
        if (l <= N) {   // structural constants of this lane's record: never rewritten
            const int r = SO(W_SD + l * SDSZ);
            if (MODEL) { sts(sm, r + SO(SD_CS + 3), 0.0); sts(sm, r + SO(SD_CE + 3), 0.0); sts(sm, r + SO(61), 0.0); }
            sts(sm, r + SO(SD_CF + 3), 0.0);                                        // psi column: (A02, A12, 1, 0) -- the 1 is set by assemble (0 for record N)
            sts(sm, r + SO(SD_CF + 8), 0.0); sts(sm, r + SO(SD_CF + 9), 0.0); sts(sm, r + SO(SD_CF + 10), 0.0);   // a column: (0,0,0,dt)
            sts(sm, r + SO(SD_CF + 15), 0.0);                                       // df column: (b0,b1,b2,0)
            sts(sm, r + SO(SD_ZERO), 0.0);
        }
        if (W == 1) syncwarp(); else block_sync();
    }

    MPC_DEV void recips(Recips& q) const {
        const double vl = isS ? L.sv - c.vLo : 1.0, vu = isS ? c.vHi - L.sv : 1.0;
        const double al = isU ? L.ua - c.aLo : 1.0, au = isU ? c.aHi - L.ua : 1.0;
        const double dl = isU ? L.ud - c.dLo : 1.0, du = isU ? c.dHi - L.ud : 1.0;
        const double h0 = rHi(0), h1 = rHi(1);
        const double r0l = isR ? L.rs[0] + h0 : 1.0, r0u = isR ? h0 - L.rs[0] : 1.0;
        const double r1l = isR ? L.rs[1] + h1 : 1.0, r1u = isR ? h1 - L.rs[1] : 1.0;
        const double pv = vl * vu, pa_ = al * au, pd_ = dl * du, p0 = r0l * r0u, p1 = r1l * r1u;
        const double pva = pv * pa_, p01 = p0 * p1, pvad = pva * pd_;
        const double iall = 1.0 / (pvad * p01);
        const double i01 = iall * pvad, ivad = iall * p01;  // 1/(p0 p1), 1/(pv pa pd)
        const double ip0 = i01 * p1, ip1 = i01 * p0;
        const double ipd = ivad * pva, iva = ivad * pd_;
        const double ipv = iva * pa_, ipa = iva * pv;
        q.vL = vu * ipv; q.vU = vl * ipv; q.aL = au * ipa; q.aU = al * ipa; q.dL = du * ipd; q.dU = dl * ipd;
        q.r0L = r0u * ip0; q.r0U = r0l * ip0; q.r1L = r1u * ip1; q.r1U = r1l * ip1;
    }

    // ------------------------------------------------------------------
    // model evaluation at the point  L + a * D  (a = 0: the current iterate) -> ev
    // ------------------------------------------------------------------
    MPC_DEV void eval_point(double a) {
        StepState D;
        ld_dx(D); ld_drs(D);
        const double sx = L.sx + a * D.dsx, sy = L.sy + a * D.dsy, sp = L.sp + a * D.dsp, sv = L.sv + a * D.dsv;
        const double ua = L.ua + a * D.dua, ud = L.ud + a * D.dud;
        const double s0 = L.rs[0] + a * D.drs[0], s1 = L.rs[1] + a * D.drs[1];
        // trig: beta = atan(r tan df) in closed form, valid for |df| < pi/2 (bounds keep |df| <= 0.5)
        EvalLane e;
        {
            const double r = c.rfrac;
            double sd, cd, sps, cps;
            mpc_sincos(ud, &sd, &cd);
            mpc_sincos(sp, &sps, &cps);
            const double Dn = cd * cd + r * r * sd * sd;
            const double iD = 1.0 / Dn;
            const double inv = sqrt(iD);
            e.cb = cd * inv;
            e.sb = r * sd * inv;
            e.cs = cps * e.cb - sps * e.sb;
            e.sn = sps * e.cb + cps * e.sb;
            e.b1 = r * iD;
            e.b2 = r * (1.0 - r * r) * (2.0 * sd * cd) * (iD * iD);
        }
        double fx = sx + c.dt * (sv * e.cs);
        const double fy = sy + c.dt * (sv * e.sn);
        double fp = sp + c.dtLb * (sv * e.sb);
        const double fv = sv + c.dt * ua;
        if (MODEL) {   // MKZMPCPathFollowerFrenet.jl:111-120: ds/dt = v cos(e_psi + beta) / (1 - e_y K(s))
            const Curv cu = curvature(sx);
            e.K = cu.K;
            e.q = 1.0 / (1.0 - sy * cu.K);
            const double g = sv * e.cs * e.q;
            fx = sx + c.dt * g;
            fp = sp + c.dt * (sv * e.sb / c.Lb - g * cu.K);
        }
        // thread k < N takes s_{k+1}; thread N takes s_0 (for the initial-condition rows); every thread u_{k-1}
        double nxt[4], prv[2];
        {
            const double dn[4] = {sx, sy, sp, sv}, up[2] = {ua, ud};
            xchg<4, 2, true>(dn, nxt, up, prv, N);
        }
        const double nx = nxt[0], ny = nxt[1], np = nxt[2], nv = nxt[3];
        if (isU) { e.rd[0] = fx - nx; e.rd[1] = fy - ny; e.rd[2] = fp - np; e.rd[3] = fv - nv; }
        else if (k == N) { e.rd[0] = cst(0) - nx; e.rd[1] = cst(1) - ny; e.rd[2] = cst(2) - np; e.rd[3] = cst(3) - nv; }
        else { e.rd[0] = e.rd[1] = e.rd[2] = e.rd[3] = 0.0; }
        const double pa = prv[0], pd = prv[1];
        const bool l0 = (k == 0);
        const double ba = l0 ? cst(5) : pa, bd = l0 ? cst(4) : pd;
        e.dr[0] = isR ? (ud - bd) - s0 : 0.0;
        e.dr[1] = isR ? (ua - ba) - s1 : 0.0;
        ev_store(e);
        // objective (MKZMPCPathFollower.jl:97-103): stage terms + rate terms counted at the later input
        double f;
        {
            const double ex = sx - ref_x(), ey = sy - ref_y(), ep = sp - ref_p(), evv = sv - cst(6);
            f = wx() * ex * ex + wy() * ey * ey + wp() * ep * ep + wv() * evv * evv;
            if (isU) {
                f += wt(6) * ua * ua + wt(7) * ud * ud;
                if (k >= 1) { const double da = ua - pa, dd = ud - pd; f += wt(4) * da * da + wt(5) * dd * dd; }
            }
        }
        double p = 1.0;
        if (isS) p *= (sv - c.vLo) * (c.vHi - sv);
        if (isU) p *= (ua - c.aLo) * (c.aHi - ua) * (ud - c.dLo) * (c.dHi - ud);
        if (isR) { const double h0 = rHi(0), h1 = rHi(1); p *= (s0 + h0) * (h0 - s0) * (s1 + h1) * (h1 - s1); }
        double lb = log(p);
        double th = fabs(e.rd[0]) + fabs(e.rd[1]) + fabs(e.rd[2]) + fabs(e.rd[3]) + fabs(e.dr[0]) + fabs(e.dr[1]);
        double r3[3] = {f, lb, th};
        treduce<OP_SUM, 3>(r3);
        ev.f = r3[0]; ev.lb = r3[1]; ev.theta = r3[2];
    }

    // scaled objective gradient at the current iterate (recomputed where needed: cheaper than six
    // doubles kept alive across the Riccati passes)
    struct Grad { double x, y, p, v, a, d; };
    MPC_DEV Grad objective_gradient() {
        Grad g;
        double nxt[2], prv[2];
        {
            const double u[2] = {L.ua, L.ud};
            xchg<2, 2, false>(u, nxt, u, prv);
        }
        const double na = nxt[0], nd = nxt[1], pa = prv[0], pd = prv[1];
        const double s2 = 2.0 * sigma;
        g.x = s2 * wx() * (L.sx - ref_x());
        g.y = s2 * wy() * (L.sy - ref_y());
        g.p = s2 * wp() * (L.sp - ref_p());
        g.v = s2 * wv() * (L.sv - cst(6));
        g.a = 0.0; g.d = 0.0;
        if (isU) {
            g.a = s2 * wt(6) * L.ua;
            g.d = s2 * wt(7) * L.ud;
            if (k >= 1) { g.a += s2 * wt(4) * (L.ua - pa); g.d += s2 * wt(5) * (L.ud - pd); }
            if (k + 1 < N) { g.a -= s2 * wt(4) * (na - L.ua); g.d -= s2 * wt(5) * (nd - L.ud); }
        }
        return g;
    }

    // MODEL 1: stage Jacobian at the current iterate (= the last evaluated point); all zero for threads without an input
    struct FJac { double a00, a01, a02, a03, a12, a13, a20, a21, a22, a23, b0, b1, b2, G0, G1, G2, G3, G4, g, K1, K2; };
    MPC_DEV FJac frenet_jac(const EvalLane& e) const {
        FJac J;
        const Curv cu = curvature(L.sx);
        const double v = L.sv, dt = isU ? c.dt : 0.0, one = isU ? 1.0 : 0.0;
        const double q2 = e.q * e.q;
        const double qs = L.sy * cu.K1 * q2, qe = e.K * q2;
        J.K1 = cu.K1; J.K2 = cu.K2;
        J.g = v * e.cs * e.q;
        J.G0 = v * e.cs * qs; J.G1 = v * e.cs * qe; J.G2 = -v * e.sn * e.q; J.G3 = e.cs * e.q; J.G4 = -v * e.sn * e.b1 * e.q;
        J.a00 = one + dt * J.G0; J.a01 = dt * J.G1; J.a02 = dt * J.G2; J.a03 = dt * J.G3; J.b0 = dt * J.G4;
        J.a12 = dt * v * e.cs; J.a13 = dt * e.sn; J.b1 = dt * v * e.cs * e.b1;
        J.a20 = -dt * (J.G0 * e.K + J.g * cu.K1); J.a21 = -dt * J.G1 * e.K; J.a22 = one - dt * J.G2 * e.K;
        J.a23 = dt * (e.sb / c.Lb - J.G3 * e.K); J.b2 = dt * (v * e.cb * e.b1 / c.Lb - J.G4 * e.K);
        return J;
    }

    // ------------------------------------------------------------------
    // Stage record assembly (lane k writes record k).
    //   req 0: least-squares multiplier system (identity Hessian, unit slack weights, zero residuals)
    //   req 1: primal-dual system, full record, residuals from `ev` (which holds the current point)
    //   req 2: primal-dual system after a change of delta_w: only the touched entries
    //   req 3: primal-dual system with the residuals already in the record (second-order correction)
    // ------------------------------------------------------------------
    MPC_DEV void assemble(int req, double mu, double dw) {
        const int r = rec();
        const Grad g = objective_gradient();
        const double gx = g.x, gy = g.y, gp = g.p, gv = g.v, ga = g.a, gd = g.d;
        EvalLane e;
        ev_load_model(e);
        BoundMult Z;
        ld_z(Z);
        double Hxx, Hyy, Hpp, Hpv = 0.0, Hvv, Hpd = 0.0, Hvd = 0.0, Haa, Hdd, Ca = 0.0, Cd = 0.0;
        double Hse = 0.0, Hsp = 0.0, Hsv = 0.0, Hsd = 0.0, Hep = 0.0, Hev = 0.0, Hed = 0.0;   // MODEL 1 only
        FJac J;
        if (MODEL) J = frenet_jac(e);
        double gsv, gua = 0.0, gud = 0.0;
        double SrW[2] = {0.0, 0.0}, br[2] = {0.0, 0.0}, wrow[2] = {0.0, 0.0}, rdr[2] = {0.0, 0.0};
        if (req == 0) {
            if (isR) for (int i = 0; i < 2; i++) { SrW[i] = 1.0; br[i] = -(Z.rvL[i] - Z.rvU[i]); wrow[i] = br[i]; }
            Hxx = Hyy = Hpp = Hvv = 1.0;
            Ca = (isU && isR) ? 1.0 : 0.0; Cd = Ca;
            Haa = 1.0 + Ca; Hdd = 1.0 + Cd;
            gsv = gv + (isS ? (-Z.zvL + Z.zvU) : 0.0);
            if (isU) { gua = ga - Z.zaL + Z.zaU; gud = gd - Z.zdL + Z.zdU; }
        } else {
            // multipliers of the rows leaving this stage (held by lane k+1)
            double y1[3];
            { const double y[3] = {L.yx, L.yy, L.yp}; xnext<3>(y, y1); }
            const double y1x = y1[0], y1y = y1[1], y1p = y1[2];
            double hpp = 0.0, hdd = 0.0, hss = 0.0, hee = 0.0;
            if (MODEL && isU) {
                // Lagrangian Hessian of the Frenet stage map over (s, e_y, e_psi, v, df): with g = v C q,
                // rows s and e_psi contribute  -dt [ (y_s - y_p K) hess g - y_p K' (e_s grad g' + grad g e_s') - y_p g K'' e_s e_s' ]
                const double v = L.sv, dt = c.dt, q = e.q, K = e.K, Cc = e.cs, Sc = e.sn, b1 = e.b1, b2 = e.b2, ey = L.sy;
                const double q2 = q * q, q3 = q2 * q, K1 = J.K1, K2 = J.K2;
                const double qs = ey * K1 * q2, qe = K * q2;
                const double qss = ey * K2 * q2 + 2.0 * ey * ey * K1 * K1 * q3, qse = K1 * q2 + 2.0 * ey * K * K1 * q3, qee = 2.0 * K * K * q3;
                const double m = y1x - y1p * K, n = y1p * K1;
                hss = -dt * (m * (v * Cc * qss) - 2.0 * n * J.G0 - y1p * J.g * K2);
                Hse = -dt * (m * (v * Cc * qse) - n * J.G1);
                Hsp = -dt * (m * (-v * Sc * qs) - n * J.G2);
                Hsv = -dt * (m * (Cc * qs) - n * J.G3);
                Hsd = -dt * (m * (-v * Sc * b1 * qs) - n * J.G4);
                hee = -dt * m * (v * Cc * qee);
                Hep = dt * m * (v * Sc * qe); Hev = -dt * m * (Cc * qe); Hed = dt * m * (v * Sc * b1 * qe);
                hpp = dt * m * (v * Cc * q) + y1y * dt * v * Sc;
                Hpv = dt * m * (Sc * q) - y1y * dt * Cc;
                Hpd = dt * m * (v * Cc * b1 * q) + y1y * dt * v * Sc * b1;
                Hvd = dt * m * (Sc * b1 * q) - y1y * dt * Cc * b1 - y1p * c.dtLb * e.cb * b1;
                hdd = dt * m * (v * q * (Cc * b1 * b1 + Sc * b2)) - y1y * dt * v * (-Sc * b1 * b1 + Cc * b2)
                      - y1p * (c.dtLb * v) * (e.cb * b2 - e.sb * b1 * b1);
            } else if (isU) {
                const double v = L.sv, dt = c.dt;
                const double e1 = y1x * e.cs + y1y * e.sn;
                const double e2 = y1x * e.sn - y1y * e.cs;
                hpp = dt * v * e1;
                Hpv = dt * e2;
                Hpd = e.b1 * hpp;
                Hvd = e.b1 * Hpv - y1p * c.dtLb * e.cb * e.b1;
                hdd = e.b1 * e.b1 * hpp + v * e.b2 * Hpv - y1p * (c.dtLb * v) * (e.cb * e.b2 - e.sb * e.b1 * e.b1);
            }
            Recips q;
            recips(q);
            // Sigma = zL/sl + zU/su ; barrier gradient b = -mu/sl + mu/su
            const double Sv = isS ? Z.zvL * q.vL + Z.zvU * q.vU : 0.0, bv = isS ? mu * (q.vU - q.vL) : 0.0;
            const double Sa = isU ? Z.zaL * q.aL + Z.zaU * q.aU : 0.0, ba = isU ? mu * (q.aU - q.aL) : 0.0;
            const double Sd = isU ? Z.zdL * q.dL + Z.zdU * q.dU : 0.0, bd = isU ? mu * (q.dU - q.dL) : 0.0;
            if (isR) {
                SrW[0] = Z.rvL[0] * q.r0L + Z.rvU[0] * q.r0U + dw; br[0] = mu * (q.r0U - q.r0L);
                SrW[1] = Z.rvL[1] * q.r1L + Z.rvU[1] * q.r1U + dw; br[1] = mu * (q.r1U - q.r1L);
                if (req == 3) { rdr[0] = lds(sm, r + SO(SD_DR)); rdr[1] = lds(sm, r + SO(SD_DR + 1)); }
                else { ev_load_resid(e); rdr[0] = e.dr[0]; rdr[1] = e.dr[1]; }
                wrow[0] = br[0] + SrW[0] * rdr[0];
                wrow[1] = br[1] + SrW[1] * rdr[1];
            }
            const double s2 = 2.0 * sigma;
            Hxx = s2 * wx() + dw; Hyy = s2 * wy() + dw; Hpp = s2 * wp() + hpp + dw; Hvv = s2 * wv() + Sv + dw;
            if (MODEL) { Hxx += hss; Hyy += hee; }
            if (isU) {
                if (k >= 1) { Ca = s2 * wt(4); Cd = s2 * wt(5); }
                if (isR) { Ca += SrW[1]; Cd += SrW[0]; }
            }
            Haa = isU ? s2 * wt(6) + Sa + dw + Ca : 1.0;
            Hdd = isU ? s2 * wt(7) + Sd + dw + Cd + hdd : 1.0;
            gsv = gv + bv;
            if (isU) { gua = ga + ba; gud = gd + bd; }
        }
        // rate-row terms: +w of the row ending at u_k, -w of the row ending at u_{k+1}
        double wn[2];
        xnext<2>(wrow, wn);
        const double wn0 = wn[0], wn1 = wn[1];
        if (isU) {
            gua += wrow[1] - ((k + 1 < N) ? wn1 : 0.0);
            gud += wrow[0] - ((k + 1 < N) ? wn0 : 0.0);
        }
        if (!isS) return;
        if (MODEL && (req == 0 || req == 1)) {
            sts2(sm, r + SO(SD_CS), J.a00, 0.0); sts(sm, r + SO(SD_CS + 2), J.a20);
            sts2(sm, r + SO(SD_CE), J.a01, isU ? 1.0 : 0.0); sts(sm, r + SO(SD_CE + 2), J.a21);
            sts2(sm, r + SO(SD_CF + 0), J.a02, J.a12); sts(sm, r + SO(SD_CF + 2), J.a22);
            sts2(sm, r + SO(SD_CF + 4), J.a03, J.a13); sts2(sm, r + SO(SD_CF + 6), J.a23, isU ? 1.0 : 0.0);
            sts(sm, r + SO(SD_CF + 11), isU ? c.dt : 0.0);
            sts2(sm, r + SO(SD_CF + 12), J.b0, J.b1); sts(sm, r + SO(SD_CF + 14), J.b2);
            sts2(sm, r + SO(SD_HSE), Hse, Hsp); sts2(sm, r + SO(SD_HSV), Hsv, Hsd); sts2(sm, r + SO(SD_HEP), Hep, Hev); sts(sm, r + SO(SD_HED), Hed);
        }
        if (req == 0 || req == 1) {
            const double A02 = isU ? -c.dt * L.sv * e.sn : 0.0, A03 = isU ? c.dt * e.cs : 0.0;
            const double A12 = isU ? c.dt * L.sv * e.cs : 0.0, A13 = isU ? c.dt * e.sn : 0.0;
            const double A23 = isU ? c.dtLb * e.sb : 0.0;
            const double b0 = A02 * e.b1, b1v = A12 * e.b1, b2v = isU ? c.dtLb * L.sv * e.cb * e.b1 : 0.0;
            const double one = isU ? 1.0 : 0.0;
            if (!MODEL) {
            sts(sm, r + SO(SD_CF + 0), A02); sts(sm, r + SO(SD_CF + 1), A12); sts(sm, r + SO(SD_CF + 2), one);
            sts(sm, r + SO(SD_CF + 4), A03); sts(sm, r + SO(SD_CF + 5), A13); sts(sm, r + SO(SD_CF + 6), A23); sts(sm, r + SO(SD_CF + 7), one);
            sts(sm, r + SO(SD_CF + 11), isU ? c.dt : 0.0);
            sts(sm, r + SO(SD_CF + 12), b0); sts(sm, r + SO(SD_CF + 13), b1v); sts(sm, r + SO(SD_CF + 14), b2v);
            }
            const bool z = (req == 0);
            ev_load_resid(e);
            sts(sm, r + SO(SD_R + 0), z ? 0.0 : e.rd[0]); sts(sm, r + SO(SD_R + 1), z ? 0.0 : e.rd[1]);
            sts(sm, r + SO(SD_R + 2), z ? 0.0 : e.rd[2]); sts(sm, r + SO(SD_R + 3), z ? 0.0 : e.rd[3]);
            sts(sm, r + SO(SD_HPV), Hpv); sts(sm, r + SO(SD_HPD), Hpd); sts(sm, r + SO(SD_HVD), Hvd);
            sts(sm, r + SO(SD_GX + 0), gx); sts(sm, r + SO(SD_GX + 1), gy); sts(sm, r + SO(SD_GX + 2), gp); sts(sm, r + SO(SD_GX + 3), gsv);
            sts(sm, r + SO(SD_BR), br[0]); sts(sm, r + SO(SD_BR + 1), br[1]);
            sts(sm, r + SO(SD_DR), rdr[0]); sts(sm, r + SO(SD_DR + 1), rdr[1]);
        }
        if (req != 3) {
            sts(sm, r + SO(SD_HXX), Hxx); sts(sm, r + SO(SD_HYY), Hyy); sts(sm, r + SO(SD_HPP), Hpp); sts(sm, r + SO(SD_HVV), Hvv);
            sts(sm, r + SO(SD_HAA), Haa); sts(sm, r + SO(SD_HDD), Hdd);
            sts(sm, r + SO(SD_CA), Ca); sts(sm, r + SO(SD_CD), Cd); sts(sm, r + SO(SD_NCA), -Ca); sts(sm, r + SO(SD_NCD), -Cd);
            sts(sm, r + SO(SD_SRW), SrW[0]); sts(sm, r + SO(SD_SRW + 1), SrW[1]);
        }
        sts(sm, r + SO(SD_GX + 4), gua); sts(sm, r + SO(SD_GX + 5), gud);
    }

    // ------------------------------------------------------------------
    // Riccati backward recursion; lanes = matrix entries.  Returns false if some stage's reduced
    // input Hessian is not positive definite (= wrong inertia of the full KKT matrix).
    //
    // Per stage s (xi = (x,y,psi,v,prev_a,prev_df), M = [A B; 0 I]):
    //   round A: TT = columns psi|v|a|df of P M, and P r + p                 (30 lanes)
    //   round B: F = H + M' (P M), f = g + M' (P r + p); idle lanes stage Ca, Cd, -Ca, -Cd  (31 lanes)
    //   round E: Fuu^{-1} (every lane), gains K, cost-to-go P <- F_xixi + F_xi,u K   (27 lanes)
    // ------------------------------------------------------------------
    MPC_DEV bool riccati_backward() {
        if (W == 1) return riccati_backward_warp();
        // long horizons: the recursion is serial in the stages, so warp 0 runs it while the other
        // warps of the team wait at the barrier that also publishes the inertia verdict
        bool ok = true;
        if ((k >> 5) == 0) ok = riccati_backward_warp();
        const int a = SO(W_XCHG + XCH_FLAG + xflip());
        if (k == 0) sts(sm, a, ok ? 1.0 : 0.0);
        block_sync();
        return lds(sm, a) != 0.0;
    }
#ifndef MPC_RICCATI_SMEM
    // Register version (MODEL 0): lane = one entry of P (21 symmetric pairs + 6 gradient entries), of P M (30 entries)
    // and of F (21 + 6); the three rounds of a stage hand their operands over with warp shuffles instead of a
    // store -> bar.warp.sync -> load round trip through shared memory.  Same arithmetic, term for term, as the
    // shared-memory version below (which MODEL 1 keeps).
    MPC_DEV bool riccati_backward_regs() {
        const int l = lane_id();
        int rl[RS_STRIDE];
        ld_roles(c.roles + 32 * role_stride_of(MODEL) + l * RS_STRIDE, rl, RS_STRIDE);
        const int a_src = launder(rl[0]), a_m = launder(rl[1]), a_mk = launder(rl[11]);
        const int b_src = launder(rl[2]), b_m = launder(rl[3]), b_mk = launder(rl[4]), b_h = launder(rl[5]);
        const int e_src = launder(rl[6]);
        const bool b_own = (launder(rl[7]) & RSF_B_OWN) != 0;
        int e_k0 = launder(rl[8]), e_k1 = launder(rl[9]);
        const int kstep = launder(rl[10]);
        double Pv;   // this lane's entry of the cost-to-go: P[i][j] (lanes 0..20), p[i] (21..26), 0 (27..31)
        {   // terminal cost-to-go from record N
            const int rN = SO(W_SD + N * SDSZ);
            int hf = SD_ZERO;
            if (l == 0) hf = SD_HXX; else if (l == 6) hf = SD_HYY; else if (l == 11) hf = SD_HPP; else if (l == 15) hf = SD_HVV;
            else if (l >= 21 && l < 25) hf = SD_GX + (l - 21);
            Pv = lds(sm, rN + SO(hf));
        }
        bool ok = true;
        int so = SO((N - 1) * SDSZ);   // byte offset of the current stage's record relative to record 0
        for (int s = N - 1; s >= 0; s--) {
            // operands from the stage record: independent of the recursion, so their loads are issued first
            const int ma = a_m + a_mk * so;
            const d2 am0 = lds2(sm, ma), am1 = lds2(sm, ma + SO(2));
            const int mb = b_m + b_mk * so;
            const d2 bm0 = lds2(sm, mb), bm1 = lds2(sm, mb + SO(2));
            const double h = lds(sm, b_h + so);
            double Tv;
            {   // ---- Round A
                const double p0 = shfl(Pv, a_src), p1 = shfl(Pv, a_src >> 5), p2 = shfl(Pv, a_src >> 10),
                             p3 = shfl(Pv, a_src >> 15), ex = shfl(Pv, a_src >> 20);
                const double t0 = p0 * am0.x + p1 * am0.y;
                const double t1 = p2 * am1.x + p3 * am1.y + ex;
                Tv = t0 + t1;
            }
            double Fv;
            {   // ---- Round B
                const double q0 = shfl(Tv, b_src), q1 = shfl(Tv, b_src >> 5), q2 = shfl(Tv, b_src >> 10),
                             q3 = shfl(Tv, b_src >> 15), x = shfl(Tv, b_src >> 20);
                const double t0 = bm0.x * q0 + bm0.y * q1 + x;
                const double t1 = bm1.x * q2 + bm1.y * q3 + h;
                Fv = b_own ? Pv + h : t0 + t1;
            }
            {   // ---- Round E (with the 2x2 inverse computed by every lane)
                const double faa = shfl(Fv, 18), fad = shfl(Fv, 19), fdd = shfl(Fv, 20);
                const double fjx = shfl(Fv, e_src >> 10), fjy = shfl(Fv, e_src >> 15);
                const double fix = shfl(Fv, e_src), fiy = shfl(Fv, e_src >> 5);
                const double f0 = shfl(Fv, e_src >> 20);
                const double det = faa * fdd - fad * fad;
                if (!(faa > 0.0) || !(det > 1e-300)) { ok = false; break; }   // (also keeps fast_rcp away from denormals)
                const double idet = fast_rcp(det);
                const double a0 = fdd * fjx - fad * fjy, a1 = faa * fjy - fad * fjx;   // adj(Fuu) (F8[j][a], F8[j][df])
                const double num = fix * a0 + fiy * a1;
                sts(sm, e_k0, -a0 * idet); sts(sm, e_k1, -a1 * idet);
                Pv = f0 - num * idet;
            }
            so -= SO(SDSZ); e_k0 -= kstep; e_k1 -= kstep;
        }
        syncwarp();   // the gains are read by other lanes (forward sweep)
        return ok;
    }
#endif
    MPC_DEV bool riccati_backward_warp() {
#ifndef MPC_RICCATI_SMEM
        if (MODEL == 0) return riccati_backward_regs();
#endif
        const int l = lane_id();
        // lane roles: shared-memory offsets of this lane's operands in the three rounds, read from the
        // table mpcb200_create computed once (riccati_roles) and laundered so that they stay in
        // registers through the stage loop instead of being rematerialised at every use
        int rl[role_stride_of(MODEL)];
        ld_roles(c.roles + l * role_stride_of(MODEL), rl, role_stride_of(MODEL));
        const int a2_p = MODEL ? launder(rl[MODEL ? 20 : 0]) : 0, a2_m = MODEL ? launder(rl[MODEL ? 21 : 0]) : 0, a2_out = MODEL ? launder(rl[MODEL ? 22 : 0]) : 0;
        const int a_p = launder(rl[0]), a_m = launder(rl[1]), a_ex = launder(rl[2]), a_out = launder(rl[3]);
        const int b_m = launder(rl[4]), b_mk = launder(rl[5]), b_t = launder(rl[6]), b_x = launder(rl[7]), b_h = launder(rl[8]);
        const int b_o1 = launder(rl[9]), b_o2 = launder(rl[10]);
        const int e_f0 = launder(rl[11]), e_fi = launder(rl[12]), e_fj = launder(rl[13]), e_o1 = launder(rl[14]), e_o2 = launder(rl[15]);
        int e_k0 = launder(rl[16]), e_k1 = launder(rl[17]);
        const int kstep = launder(rl[18]);
        {   // terminal cost-to-go from record N
            const int rN = SO(W_SD + N * SDSZ);
            for (int e = l; e < 36; e += 32) {
                const int i = e / 6, j = e - 6 * i;
                double v = 0.0;
                if (i == j && i < 4) v = lds(sm, rN + SO((i == 0) ? SD_HXX : (i == 1) ? SD_HYY : (i == 2) ? SD_HPP : SD_HVV));
                sts(sm, SO(W_P + e), v);
            }
            if (l < 6) sts(sm, SO(W_PV + l), (l < 4) ? lds(sm, rN + SO(SD_GX + l)) : 0.0);
        }
        syncwarp();
        bool ok = true;
        int so = SO((N - 1) * SDSZ);   // byte offset of the current stage's record relative to record 0
        for (int s = N - 1; s >= 0; s--) {
            {   // ---- Round A
                const d2 p0 = lds2(sm, a_p), p1 = lds2(sm, a_p + SO(2));
                const int m = a_m + so;
                const d2 m0 = lds2(sm, m), m1 = lds2(sm, m + SO(2));
                const double ex = lds(sm, a_ex);
                const double t0 = p0.x * m0.x + p0.y * m0.y;
                const double t1 = p1.x * m1.x + p1.y * m1.y + ex;
                sts(sm, a_out, t0 + t1);
                if (MODEL) {   // second task: columns s | e_y of P M (lanes 0..11; the others write the sink)
                    const d2 u0 = lds2(sm, a2_p), u1 = lds2(sm, a2_p + SO(2));
                    const int m2 = a2_m + so;
                    const d2 w0 = lds2(sm, m2), w1 = lds2(sm, m2 + SO(2));
                    sts(sm, a2_out, (u0.x * w0.x + u0.y * w0.y) + (u1.x * w1.x + u1.y * w1.y));
                }
            }
            syncwarp();
            {   // ---- Round B
                const int m = b_m + b_mk * so;
                const d2 m0 = lds2(sm, m), m1 = lds2(sm, m + SO(2));
                const d2 q0 = lds2(sm, b_t), q1 = lds2(sm, b_t + SO(2));
                const double x = lds(sm, b_x);
                const double h = lds(sm, b_h + so);
                const double t0 = m0.x * q0.x + m0.y * q0.y + x;
                const double t1 = m1.x * q1.x + m1.y * q1.y + h;
                const double o = t0 + t1;
                sts(sm, b_o1, o); sts(sm, b_o2, o);
            }
            syncwarp();
            {   // ---- Round E (with the 2x2 inverse computed by every lane)
                const d2 fa = lds2(sm, SO(W_F + 28));
                const double fdd = lds(sm, SO(W_F + 35));
                const d2 fj = lds2(sm, e_fj);
                const d2 fi = lds2(sm, e_fi);
                const double f0 = lds(sm, e_f0);
                const double faa = fa.x, fad = fa.y;
                const double det = faa * fdd - fad * fad;
                if (!(faa > 0.0) || !(det > 1e-300)) { ok = false; break; }   // (also keeps fast_rcp away from denormals)
                // Fuu^{-1} = adj(Fuu) / det: everything that does not need 1/det is computed while the
                // reciprocal is in flight, so only one multiply-add follows it
                const double idet = fast_rcp(det);
                const double a0 = fdd * fj.x - fad * fj.y, a1 = faa * fj.y - fad * fj.x;   // adj(Fuu) (F8[j][a], F8[j][df])
                const double num = fi.x * a0 + fi.y * a1;
                sts(sm, e_k0, -a0 * idet); sts(sm, e_k1, -a1 * idet);
                const double o = f0 - num * idet;
                sts(sm, e_o1, o); sts(sm, e_o2, o);
            }
            syncwarp();
            so -= SO(SDSZ); e_k0 -= kstep; e_k1 -= kstep;
        }
        return ok;
    }

    // forward sweep: one scalar recursion per problem.  Eight lanes of one warp run it (a quarter
    // warp: every broadcast shared-memory load is one wavefront instead of four) and write each
    // stage's step straight into that stage's per-thread fields.
    MPC_DEV void riccati_forward() {
        if (lane_id() < 8 && (W == 1 || (k >> 5) == 0)) {
            int kp = SO(W_SD + (N + 1) * SDSZ);
            int r = SO(W_SD);
            int fa = SO(lf_offset(N, MODEL) + G_DX_OFF * (N + 2));   // step group of stage 0
            const d2 i01 = lds2(sm, SO(W_SD + N * SDSZ + SD_R)), i23 = lds2(sm, SO(W_SD + N * SDSZ + SD_R + 2));  // ds_0
            double s0 = i01.x, s1 = i01.y, s2 = i23.x, s3 = i23.y;
            double pa = 0.0, pd = 0.0;
            // The recursion is one dependent chain per problem (s -> u -> next s).  The gains of a stage are what the
            // chain needs first, so they are loaded one stage ahead (while the previous stage's next-state sums run);
            // the record columns are needed only after the inputs, so their loads, issued at the top, are covered by
            // the input sums.
            d2 ka0 = lds2(sm, kp), ka1 = lds2(sm, kp + SO(2)), ka2 = lds2(sm, kp + SO(4)), kx = lds2(sm, kp + SO(6));
            d2 kd0 = lds2(sm, kp + SO(8)), kd1 = lds2(sm, kp + SO(10)), kd2 = lds2(sm, kp + SO(12));
            const int kp_last = kp + (N - 1) * SO(KST_STRIDE);
            for (int s = 0; s < N; s++) {
                const d2 cp = lds2(sm, r + SO(SD_CF + 0)), cv = lds2(sm, r + SO(SD_CF + 4)), cd = lds2(sm, r + SO(SD_CF + 12));
                const double a23 = lds(sm, r + SO(SD_CF + 6)), b2 = lds(sm, r + SO(SD_CF + 14));
                const d2 r01 = lds2(sm, r + SO(SD_R)), r23 = lds2(sm, r + SO(SD_R + 2));
                double a00 = 0.0, a20 = 0.0, a01 = 0.0, a21 = 0.0, a22 = 0.0;
                if (MODEL) {   // dense s and e_y columns; the unit parts are in the record
                    a00 = lds(sm, r + SO(SD_CS)); a20 = lds(sm, r + SO(SD_CS + 2));
                    a01 = lds(sm, r + SO(SD_CE)); a21 = lds(sm, r + SO(SD_CE + 2)); a22 = lds(sm, r + SO(SD_CF + 2));
                }
                // the terms that do not need the values produced last (s0..s3 for the inputs, the inputs for the next
                // state) are summed first
                const double ua = ((ka2.x * pa + ka2.y * pd) + kx.x) + ((ka0.x * s0 + ka0.y * s1) + (ka1.x * s2 + ka1.y * s3));
                const double ud = ((kd1.y * pa + kd2.x * pd) + kd2.y) + ((kx.y * s0 + kd0.x * s1) + (kd0.y * s2 + kd1.x * s3));
                sts2(sm, fa, s0, s1); sts2(sm, fa + SO(2), s2, s3); sts2(sm, fa + SO(4), ua, ud);
                kp += SO(KST_STRIDE);
                {   // gains of the next stage (the last stage re-reads its own: no access past the gain area)
                    const int kn = (kp <= kp_last) ? kp : kp_last;
                    ka0 = lds2(sm, kn); ka1 = lds2(sm, kn + SO(2)); ka2 = lds2(sm, kn + SO(4)); kx = lds2(sm, kn + SO(6));
                    kd0 = lds2(sm, kn + SO(8)); kd1 = lds2(sm, kn + SO(10)); kd2 = lds2(sm, kn + SO(12));
                }
                double n0 = ((s0 + r01.x) + (cp.x * s2 + cv.x * s3)) + cd.x * ud;
                double n1 = ((s1 + r01.y) + (cp.y * s2 + cv.y * s3)) + cd.y * ud;
                double n2 = ((s2 + r23.x) + a23 * s3) + b2 * ud;
                const double n3 = (s3 + r23.y) + c.dt * ua;
                if (MODEL) {
                    n0 = (r01.x + (a00 * s0 + a01 * s1)) + ((cp.x * s2 + cv.x * s3) + cd.x * ud);
                    n1 = ((s1 + r01.y) + (cp.y * s2 + cv.y * s3)) + cd.y * ud;
                    n2 = (r23.x + (a20 * s0 + a21 * s1)) + ((a22 * s2 + a23 * s3) + b2 * ud);
                }
                s0 = n0; s1 = n1; s2 = n2; s3 = n3; pa = ua; pd = ud;
                r += SO(SDSZ); fa += SO(G_DX_STRIDE);
            }
            sts2(sm, fa, s0, s1); sts2(sm, fa + SO(2), s2, s3); sts2(sm, fa + SO(4), 0.0, 0.0);
        }
        tsync();
    }

    // new equality multipliers from stationarity in the state variables (parallel suffix sums),
    // new rate-row multipliers and slack steps; the condensed blocks are read back from the record
    MPC_DEV void recover_duals() {
        const int r = rec();
        StepState D;
        ld_dx(D);
        double lx = 0.0, ly = 0.0, lp = 0.0, lv = 0.0;
        const double hpv = lds(sm, r + SO(SD_HPV));
        if (isS) {
            lx = -(lds(sm, r + SO(SD_HXX)) * D.dsx + lds(sm, r + SO(SD_GX)));
            ly = -(lds(sm, r + SO(SD_HYY)) * D.dsy + lds(sm, r + SO(SD_GX + 1)));
            lp = -(lds(sm, r + SO(SD_HPP)) * D.dsp + hpv * D.dsv + lds(sm, r + SO(SD_HPD)) * D.dud + lds(sm, r + SO(SD_GX + 2)));
            lv = -(hpv * D.dsp + lds(sm, r + SO(SD_HVV)) * D.dsv + lds(sm, r + SO(SD_HVD)) * D.dud + lds(sm, r + SO(SD_GX + 3)));
        }
        double prv[2];
        if (MODEL) {
            // the s and e_y columns of A are dense: no suffix sums; costate recursion  lambda_k = l_k + A_k' lambda_{k+1}
            // run serially by one thread, in place, through the multiplier group
            if (isS) {
                const d2 h0 = lds2(sm, r + SO(SD_HSE)), h1 = lds2(sm, r + SO(SD_HSV)), h2 = lds2(sm, r + SO(SD_HEP));
                const double hed = lds(sm, r + SO(SD_HED));
                lx -= h0.x * D.dsy + h0.y * D.dsp + h1.x * D.dsv + h1.y * D.dud;
                ly -= h0.x * D.dsx + h2.x * D.dsp + h2.y * D.dsv + hed * D.dud;
                lp -= h0.y * D.dsx + h2.x * D.dsy;
                lv -= h1.x * D.dsx + h2.y * D.dsy;
            }
            D.nyx = lx; D.nyy = ly; D.nyp = lp; D.nyv = lv; D.nyd[0] = D.nyd[1] = 0.0;
            st_dy(D);
            tsync();
            if (k == 0) {
                int ya = SO(lf_offset(N, MODEL) + G_DY_OFF * (N + 2)) + N * SO(G_DY_STRIDE);   // multiplier group of stage N
                int rr = SO(W_SD + (N - 1) * SDSZ);
                d2 y01 = lds2(sm, ya), y23 = lds2(sm, ya + SO(2));
                for (int s = N - 1; s >= 0; s--) {
                    ya -= SO(G_DY_STRIDE);
                    const d2 l01 = lds2(sm, ya), l23 = lds2(sm, ya + SO(2));
                    const double a00 = lds(sm, rr + SO(SD_CS)), a20 = lds(sm, rr + SO(SD_CS + 2));
                    const double a01 = lds(sm, rr + SO(SD_CE)), a21 = lds(sm, rr + SO(SD_CE + 2));
                    const d2 cp = lds2(sm, rr + SO(SD_CF + 0)), cv = lds2(sm, rr + SO(SD_CF + 4));
                    const double a22 = lds(sm, rr + SO(SD_CF + 2)), a23 = lds(sm, rr + SO(SD_CF + 6));
                    const double m0 = l01.x + (a00 * y01.x + a20 * y23.x);
                    const double m1 = l01.y + ((a01 * y01.x + y01.y) + a21 * y23.x);
                    const double m2 = l23.x + ((cp.x * y01.x + cp.y * y01.y) + a22 * y23.x);
                    const double m3 = l23.y + ((cv.x * y01.x + cv.y * y01.y) + (a23 * y23.x + y23.y));
                    y01.x = m0; y01.y = m1; y23.x = m2; y23.y = m3;
                    sts2(sm, ya, m0, m1); sts2(sm, ya + SO(2), m2, m3);
                    rr -= SO(SDSZ);
                }
            }
            tsync();
            ld_dy(D);
            { const double du[2] = {D.dua, D.dud}; xprev<2>(du, prv); }
        } else {
        const double hasn = isU ? 1.0 : 0.0;
        const d2 c0 = lds2(sm, r + SO(SD_CF + 0)), c1 = lds2(sm, r + SO(SD_CF + 4));   // (A02, A12), (A03, A13)
        const double A23 = lds(sm, r + SO(SD_CF + 6));
        double lxy[2] = {lx, ly}, n1[2];
        tsuffix<2>(lxy);   // y_x, y_y: two interleaved suffix sums
        D.nyx = lxy[0]; D.nyy = lxy[1];
        xnext<2>(lxy, n1);
        const double nx1 = n1[0], ny1 = n1[1];
        double t1 = lp + hasn * (c0.x * nx1 + c0.y * ny1);
        tsuffix<1>(&t1);
        D.nyp = t1;
        double np1;
        { const double du[2] = {D.dua, D.dud}; xchg<1, 2, false>(&t1, &np1, du, prv); }
        t1 = lv + hasn * (c1.x * nx1 + c1.y * ny1 + A23 * np1);
        tsuffix<1>(&t1);
        D.nyv = t1;
        }
        const double pa = prv[0], pd = prv[1];
        D.drs[0] = D.drs[1] = 0.0; D.nyd[0] = D.nyd[1] = 0.0;
        if (isR) {
            const double ba = (k == 0) ? 0.0 : pa, bd = (k == 0) ? 0.0 : pd;
            const d2 srw = lds2(sm, r + SO(SD_SRW)), brr = lds2(sm, r + SO(SD_BR)), drr = lds2(sm, r + SO(SD_DR));
            D.drs[0] = (D.dud - bd) + drr.x;
            D.drs[1] = (D.dua - ba) + drr.y;
            D.nyd[0] = srw.x * D.drs[0] + brr.x;
            D.nyd[1] = srw.y * D.drs[1] + brr.y;
        }
        st_drs(D); st_dy(D);
    }

    // fraction-to-the-boundary for the primal step: tau / max_i( -dx_i / slack_i ), division-free per element
    MPC_DEV double alpha_primal(double tau) {
        StepState D;
        ld_dx(D); ld_drs(D);
        double num = 0.0, den = 1.0;   // largest ratio num/den (num >= 0, den > 0) by cross-multiplication
        auto upd = [&](double dx, double sl, double su) {
            const double n = fabs(dx), d = (dx < 0.0) ? sl : su;
            if (n * den > num * d) { num = n; den = d; }
        };
        if (isS) upd(D.dsv, L.sv - c.vLo, c.vHi - L.sv);
        if (isU) { upd(D.dua, L.ua - c.aLo, c.aHi - L.ua); upd(D.dud, L.ud - c.dLo, c.dHi - L.ud); }
        if (isR) { const double h0 = rHi(0), h1 = rHi(1); upd(D.drs[0], L.rs[0] + h0, h0 - L.rs[0]); upd(D.drs[1], L.rs[1] + h1, h1 - L.rs[1]); }
        const double a = (num > 0.0) ? tau * den / num : 1.0;  // num == 0: no limit from this lane
        return dmin_(1.0, tmin(a));
    }

    // ------------------------------------------------------------------
    // Restoration by rollout (oracle: ipm_rollout_restore).  The inputs of the current iterate are
    // projected stage by stage onto the input box, the rate rows and the speed bounds, and the states
    // are rolled out from the measured state (MKZMPCPathFollower.jl:115-123).  One serial recursion
    // per problem, run by one thread through the per-thread step fields (dead at this point).
    // ------------------------------------------------------------------
    MPC_DEV void rollout_restore() {
        {
            StepState D;
            D.dsx = D.dsy = D.dsp = D.dsv = 0.0; D.dua = L.ua; D.dud = L.ud;
            st_dx(D);
        }
        tsync();
        if (k == 0) {   // one thread: the recursion reads and rewrites the same words stage by stage
            RolloutConsts rc;
            rc.dt = c.dt; rc.dtc = c.dtc; rc.dtLb = c.dtLb; rc.rfrac = c.rfrac; rc.vmin = c.vmin; rc.vmax = c.vmax;
            rc.amax = c.amax; rc.smax = c.smax; rc.admax = c.admax; rc.sdmax = c.sdmax;
            rc.model = MODEL; rc.kp[0] = rc.kp[1] = rc.kp[2] = rc.kp[3] = 0.0;
            if (MODEL) { const int a = grp(G_REF_OFF, 4); rc.kp[0] = lds(sm, a); rc.kp[1] = lds(sm, a + SO(1)); rc.kp[2] = lds(sm, a + SO(2)); rc.kp[3] = lds(sm, a + SO(3)); }
            rollout_core(sm, SO(lf_offset(N, MODEL) + G_DX_OFF * (N + 2)), SO(W_CONST), N, rc);
        }
        tsync();
        if (isS) {
            StepState D;
            ld_dx(D);
            L.sx = D.dsx; L.sy = D.dsy; L.sp = D.dsp; L.sv = D.dsv; L.ua = D.dua; L.ud = D.dud;
        }
    }

    // np.argmin of the squared distance to (X, Y) over all samples of the path (ref_gps_traj.py:136-137; first index on ties),
    // each distance rounded operation by operation like numpy's.  Not a scan of all samples: a chunk of PATH_CHUNK consecutive
    // samples whose bounding circle lies further away than the far side of the nearest circle cannot hold the minimum (margins
    // far above the rounding of the bounds), so a lane scans only those of its chunks that can -- usually the two or three
    // around the vehicle, spread over as many lanes.  A pose that is not finite gives index 0, like argmin of an all-NaN array.
    MPC_DEV int nearest_sample(const PathTable& p, double X, double Y) {
        double bd = 1e300; int bi = 0x7fffffff;
        double ub = 1e300;
        if (p.cb) {
            const double *cx = p.cb, *cy = p.cb + p.nch, *cr = p.cb + 2 * p.nch;
            for (int c = k; c < p.nch; c += 32 * W) {
                const double dx = cx[c] - X, dy = cy[c] - Y, u = sqrt(dx * dx + dy * dy) + cr[c];
                if (u < ub) ub = u;
            }
            ub = tmin(ub);
        }
        if (ub < 1e300) {
            const double *cx = p.cb, *cy = p.cb + p.nch, *cr = p.cb + 2 * p.nch;
            const double thr = ub * (1.0 + 1e-9) + 1e-9 + 1e-12 * (fabs(X) + fabs(Y));
            for (int c = k; c < p.nch; c += 32 * W) {
                const double cdx = cx[c] - X, cdy = cy[c] - Y;
                if (sqrt(cdx * cdx + cdy * cdy) - cr[c] > thr) continue;
                const int i0 = c * PATH_CHUNK, i1 = (i0 + PATH_CHUNK < p.n) ? i0 + PATH_CHUNK : p.n;
                for (int i = i0; i < i1; i++) {
                    const double dx = p.X[i] - X, dy = p.Y[i] - Y, d = add_rn(mul_rn(dx, dx), mul_rn(dy, dy));
                    if (d < bd) { bd = d; bi = i; }
                }
            }
        } else {
            for (int i = k; i < p.n; i += 32 * W) {
                const double dx = p.X[i] - X, dy = p.Y[i] - Y, d = add_rn(mul_rn(dx, dx), mul_rn(dy, dy));
                if (d < bd) { bd = d; bi = i; }
            }
        }
        targmin(bd, bi);
        return (bi < p.n) ? bi : 0;
    }

    // get_waypoints (ref_gps_traj.py:131-218) for the whole team: thread k returns waypoint k (k <= N); returns stop_cmd.
    // Nearest sample over the whole path (:136-137), np.interp of X, Y, psi at t_closest + k dt -- or at
    // s_closest + (k + 1) dt v_target in distance mode (:175) --, heading unwrap (:204-218), stop_cmd (:198-200).
    MPC_DEV bool get_waypoints(const PathTable& p, double traj_dt, double X, double Y, double yaw, bool use_vtarget,
                               double v_target, double& xr, double& yr, double& pr) {
        const int bi = nearest_sample(p, X, Y);
        const double* absc = use_vtarget ? p.s : p.t;
        const double start = absc[bi];
        xr = yr = pr = 0.0;
        if (k <= N) {
            const double q = use_vtarget ? add_rn(mul_rn(mul_rn((double)(k + 1), traj_dt), v_target), start)
                                         : add_rn(mul_rn((double)k, traj_dt), start);
            xr = np_interp(q, absc, p.X, p.n); yr = np_interp(q, absc, p.Y, p.n); pr = np_interp(q, absc, p.psi, p.n);
        }
        // heading wrap-around fix (:204-218)
        const double PI = 3.141592653589793;
        double nxt;
        xnext<1>(&pr, &nxt);
        double c12[2] = {(k < N) ? fabs(nxt - pr) : 0.0, (k <= N) ? fabs(pr - yaw) : 0.0};
        treduce<OP_MAX, 2>(c12);
        if (!(c12[0] < PI && c12[1] < PI)) {
            const double a0 = pr, a1 = pr + 2.0 * PI, a2 = pr - 2.0 * PI;
            double b = a0, e = fabs(a0 - yaw);
            if (fabs(a1 - yaw) < e) { e = fabs(a1 - yaw); b = a1; }
            if (fabs(a2 - yaw) < e) { b = a2; }
            pr = b;
        }
        const double lx = bcast_from(xr, N), ly = bcast_from(yr, N);
        return lx == p.X[p.n - 1] && ly == p.Y[p.n - 1];
    }

    MPC_DEV bool nlp_feasible() const {
        const double e = 1e-8;
        const double lim_d = c.sdmax * c.dtc, lim_a = c.admax * c.dtc;
        const double v0 = cst(3), up0 = cst(4), up1 = cst(5);
        if (v0 < c.vmin - e * dmax_(1.0, fabs(c.vmin))) return false;
        if (v0 > c.vmax + e * dmax_(1.0, fabs(c.vmax))) return false;
        if (up0 - lim_d > c.smax + 2 * e || up0 + lim_d < -c.smax - 2 * e) return false;
        if (up1 - lim_a > c.amax + 2 * e || up1 + lim_a < -c.amax - 2 * e) return false;
        return true;
    }

    // ------------------------------------------------------------------
    // the whole solve
    // ------------------------------------------------------------------
    MPC_DEV Result solve() {
        Result res; res.status = 4; res.iters = 0; res.cost = 0.0;
        L.rs[0] = L.rs[1] = 0.0;
        L.ryd[0] = L.ryd[1] = 0.0; L.yx = L.yy = L.yp = L.yv = 0.0;

        const bool feasible = nlp_feasible();
        int ret = feasible ? -1 : 2;

        // ---- objective scaling from the gradient at the user's start point
        sigma = 1.0;
        {
            const Grad g = objective_gradient();
            double gm = dmax_(dmax_(fabs(g.x), fabs(g.y)), dmax_(fabs(g.p), fabs(g.v)));
            gm = tmax(dmax_(gm, dmax_(fabs(g.a), fabs(g.d))));
            sigma = (gm > K_SCALE_MAX_GRAD) ? dmax_(K_SCALE_MAX_GRAD / gm, 1e-8) : 1.0;
        }
        enum { PH_INIT = 0, PH_EVAL0, PH_LS, PH_BEGIN, PH_PD, PH_RESOLVE_EVAL, PH_RESOLVE, PH_TRIAL, PH_SOC, PH_RESTO };
        int phase = PH_INIT;
        bool do_solve = false, do_eval = false, eval_ftb = false;
        bool resto_check = false, cur_acceptable = false, had_acceptable = false;
        int n_resto = 0;
        int req = 0;
        double ev_alpha = 0.0;

        double mu = K_MU_INIT, tau = dmax_(K_TAU_MIN, 1.0 - K_MU_INIT);
        double dw = 0.0, dw_last = 0.0, theta_max = -1.0, theta_min = -1.0;
        double f_phi = 0.0, f_theta = 0.0;  // this lane's filter entry (entry e lives in lane e)
        int nfilt = 0, accept_count = 0, iter = 0;
        bool tiny_last = false, tiny = false, solve_ok = false;
        // current-point scalars and line-search state of the current iteration
        double cur_theta = 0.0, cur_f = 0.0, cur_lb = 0.0;
        double phi = 0.0, gBd = 0.0, alpha = 1.0, alpha_max = 1.0, Rft = 0.0, a_soc = 0.0;
        double th_soc_old = 0.0;
        int nsteps = 0, soc_cnt = 0;
        const int nz = 2 * (3 * N + 1) + 4 * (N - 1);  // bound multipliers: x-bounds + slack bounds
        const int my = 4 * (N + 1) + 2 * (N - 1);      // equality multipliers y_c, y_d

        while (feasible) {
            // ================= shared heavy work =================
            if (do_solve) {
                assemble(req, mu, dw);
                tsync();
                solve_ok = riccati_backward();
                if (solve_ok) { riccati_forward(); recover_duals(); }
                tsync();
            }
            if (do_eval) {
                if (eval_ftb) { ev_alpha = alpha_primal(tau); a_soc = ev_alpha; }
                eval_point(ev_alpha);
            }
            do_solve = false; do_eval = false; eval_ftb = false;

            // ================= driver =================
            if (phase == PH_TRIAL || phase == PH_SOC) {
                const double alpha_test = (phase == PH_SOC) ? alpha_max : alpha;
                const double th_t = ev.theta;
                const double ph_t = sigma * ev.f - mu * ev.lb;
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
                    const bool mine = (k >= nfilt) || cmp_le(ph_t, f_phi, f_phi) || cmp_le(th_t, f_theta, f_theta);
                    ok = tall(mine) && ok;
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
                        // c_soc <- a_soc * c_soc + c(trial), accumulated in the record's right-hand-side fields
                        th_soc_old = th_t;
                        if (isS) {
                            const int r = rec();
                            EvalLane e;
                            ev_load_resid(e);
                            for (int i = 0; i < 4; i++) sts(sm, r + SO(SD_R + i), a_soc * lds(sm, r + SO(SD_R + i)) + e.rd[i]);
                            sts(sm, r + SO(SD_DR), a_soc * lds(sm, r + SO(SD_DR)) + e.dr[0]);
                            sts(sm, r + SO(SD_DR + 1), a_soc * lds(sm, r + SO(SD_DR + 1)) + e.dr[1]);
                        }
                        tsync();
                        phase = PH_SOC; do_solve = true; req = 3; do_eval = true; eval_ftb = true;
                        continue;
                    }
                    if (phase == PH_SOC) {
                        // corrections exhausted: re-evaluate the current point, recompute the Newton direction, backtrack
                        phase = PH_RESOLVE_EVAL; do_eval = true; ev_alpha = 0.0;
                        {
                            StepState D;
                            D.dsx = D.dsy = D.dsp = D.dsv = D.dua = D.dud = 0.0; D.drs[0] = D.drs[1] = 0.0;
                            st_dx(D); st_drs(D);
                        }
                        continue;
                    }
                    // plain backtracking
                    double alpha_min = K_GAMMA_THETA;
                    if (gBd < 0.0) alpha_min = dmin_(K_GAMMA_THETA, K_GAMMA_PHI * theta / (-gBd));
                    alpha_min *= K_ALPHA_MIN_FRAC;
                    alpha *= 0.5; nsteps++;
                    bool above_min = alpha > alpha_min;   // alpha > alpha_min_frac * min(gamma_theta, gamma_phi theta / -gBd, delta R)
                    if (!above_min && gBd < 0.0 && theta <= theta_min)
                        above_min = ratio_test(1, alpha, K_ALPHA_MIN_FRAC * (K_DELTA * Rft), theta, -gBd);
                    if (!above_min) {   // Ipopt would enter the restoration phase ...
                        if (cur_acceptable) { ret = 1; break; }   // ... unless the point is acceptable: Solved_To_Acceptable_Level
                        if (cur_theta <= 1e-2 * c.tol) { ret = had_acceptable ? 1 : -2; break; }   // ... or almost feasible (see oracle)
                        if (n_resto < K_MAX_RESTO) { phase = PH_RESTO; continue; }
                        ret = -2; break;
                    }
                    ev_alpha = alpha; do_eval = true; phase = PH_TRIAL;
                    continue;
                }
                // ---------------- accepted ----------------
                if (phase == PH_SOC) alpha = a_soc;
                if (!tiny && !(ftype && arm) && nfilt < NFILT_MAX) {
                    if (k == nfilt) { f_phi = phi - K_GAMMA_PHI * theta; f_theta = (1.0 - K_GAMMA_THETA) * theta; }
                    nfilt++;
                }
                {
                    // bound-multiplier steps from the accepted direction: dz = (mu -/+ z dx)/slack - z
                    StepState D;
                    ld_dx(D); ld_drs(D); ld_dy(D);
                    BoundMult Z;
                    ld_z(Z);
                    Recips q;
                    recips(q);
                    double dzvL = 0, dzvU = 0, dzaL = 0, dzaU = 0, dzdL = 0, dzdU = 0, drvL[2] = {0, 0}, drvU[2] = {0, 0};
                    if (isS) { dzvL = (mu - Z.zvL * D.dsv) * q.vL - Z.zvL; dzvU = (mu + Z.zvU * D.dsv) * q.vU - Z.zvU; }
                    if (isU) {
                        dzaL = (mu - Z.zaL * D.dua) * q.aL - Z.zaL; dzaU = (mu + Z.zaU * D.dua) * q.aU - Z.zaU;
                        dzdL = (mu - Z.zdL * D.dud) * q.dL - Z.zdL; dzdU = (mu + Z.zdU * D.dud) * q.dU - Z.zdU;
                    }
                    if (isR) {
                        drvL[0] = (mu - Z.rvL[0] * D.drs[0]) * q.r0L - Z.rvL[0]; drvU[0] = (mu + Z.rvU[0] * D.drs[0]) * q.r0U - Z.rvU[0];
                        drvL[1] = (mu - Z.rvL[1] * D.drs[1]) * q.r1L - Z.rvL[1]; drvU[1] = (mu + Z.rvU[1] * D.drs[1]) * q.r1U - Z.rvU[1];
                    }
                    double num = 0.0, den = 1.0;   // dual fraction-to-the-boundary: largest -dz/z by cross-multiplication
                    auto lim = [&](double z, double dz) { if (dz < 0.0 && -dz * den > num * z) { num = -dz; den = z; } };
                    lim(Z.zvL, dzvL); lim(Z.zvU, dzvU); lim(Z.zaL, dzaL); lim(Z.zaU, dzaU); lim(Z.zdL, dzdL); lim(Z.zdU, dzdU);
                    lim(Z.rvL[0], drvL[0]); lim(Z.rvU[0], drvU[0]); lim(Z.rvL[1], drvL[1]); lim(Z.rvU[1], drvU[1]);
                    const double az = dmin_(1.0, tmin(num > 0.0 ? tau * den / num : 1.0));
                    // primal, equality multipliers (primal step size), bound multipliers (dual step size)
                    L.sx += alpha * D.dsx; L.sy += alpha * D.dsy; L.sp += alpha * D.dsp; L.sv += alpha * D.dsv;
                    L.ua += alpha * D.dua; L.ud += alpha * D.dud; L.rs[0] += alpha * D.drs[0]; L.rs[1] += alpha * D.drs[1];
                    L.yx += alpha * (D.nyx - L.yx); L.yy += alpha * (D.nyy - L.yy); L.yp += alpha * (D.nyp - L.yp); L.yv += alpha * (D.nyv - L.yv);
                    L.ryd[0] += alpha * (D.nyd[0] - L.ryd[0]); L.ryd[1] += alpha * (D.nyd[1] - L.ryd[1]);
                    // z += az dz, then the kappa_sigma safeguard z in [mu / (kappa s), kappa mu / s].  The test is
                    // division-free; the clamp itself (two divisions per multiplier) is rare and kept out of
                    // line so that it does not sit, ten times over, in the middle of the hot path.
                    bool clamp = false;
                    auto upd = [&](double& z, double dz, double sl) {
                        z += az * dz;
                        const double pz = z * sl;
                        clamp = clamp || (pz > K_KAPPA_SIGMA * mu) || (pz * K_KAPPA_SIGMA < mu);
                    };
                    const double h0 = rHi(0), h1 = rHi(1);
                    if (isS) { upd(Z.zvL, dzvL, L.sv - c.vLo); upd(Z.zvU, dzvU, c.vHi - L.sv); }
                    if (isU) {
                        upd(Z.zaL, dzaL, L.ua - c.aLo); upd(Z.zaU, dzaU, c.aHi - L.ua);
                        upd(Z.zdL, dzdL, L.ud - c.dLo); upd(Z.zdU, dzdU, c.dHi - L.ud);
                    }
                    if (isR) {
                        upd(Z.rvL[0], drvL[0], L.rs[0] + h0); upd(Z.rvU[0], drvU[0], h0 - L.rs[0]);
                        upd(Z.rvL[1], drvL[1], L.rs[1] + h1); upd(Z.rvU[1], drvU[1], h1 - L.rs[1]);
                    }
                    if (clamp) {
                        double zz[10] = {Z.zvL, Z.zvU, Z.zaL, Z.zaU, Z.zdL, Z.zdU, Z.rvL[0], Z.rvU[0], Z.rvL[1], Z.rvU[1]};
                        const double sl[10] = {L.sv - c.vLo, c.vHi - L.sv, L.ua - c.aLo, c.aHi - L.ua, L.ud - c.dLo, c.dHi - L.ud,
                                               L.rs[0] + h0, h0 - L.rs[0], L.rs[1] + h1, h1 - L.rs[1]};
                        kappa_sigma_clamp(zz, sl, mu);
                        Z.zvL = zz[0]; Z.zvU = zz[1]; Z.zaL = zz[2]; Z.zaU = zz[3]; Z.zdL = zz[4]; Z.zdU = zz[5];
                        Z.rvL[0] = zz[6]; Z.rvU[0] = zz[7]; Z.rvL[1] = zz[8]; Z.rvU[1] = zz[9];
                    }
                    st_z(Z);
                }
                // the accepted trial evaluation (in ev) is the next iteration's current evaluation
                cur_theta = ev.theta; cur_f = ev.f; cur_lb = ev.lb;
                tiny_last = tiny;
                iter++;
                phase = PH_BEGIN;
            }
#ifdef MPC_TRACE
            if (phase == PH_RESTO && k == 0) printf("   RESTO at it %d: alpha %.3e gBd %.3e theta %.3e acceptable %d nsteps %d\n", iter, alpha, gBd, cur_theta, (int)cur_acceptable, nsteps);
#endif
            if (phase == PH_RESTO) {
                // The line search failed where Ipopt would enter its restoration phase.  That phase is
                // not restated; instead the iterate is replaced by the rollout of its own (projected)
                // inputs, which satisfies the equality rows by construction, and the iteration is
                // re-initialised there with mu and the filter kept (oracle: ipm_rollout_restore).
                n_resto++; had_acceptable = false;
                if (nfilt < NFILT_MAX) {   // PrepareRestoPhaseStart: the point that is left enters the filter
                    if (k == nfilt) { f_phi = phi - K_GAMMA_PHI * cur_theta; f_theta = (1.0 - K_GAMMA_THETA) * cur_theta; }
                    nfilt++;
                }
                rollout_restore();
                L.yx = L.yy = L.yp = L.yv = 0.0; L.ryd[0] = L.ryd[1] = 0.0;
                resto_check = true; tiny_last = false;
                iter++;
                phase = PH_INIT;
            }
            if (phase == PH_INIT) {
                // ---- interior start from the primal point in L (DefaultIterateInitializer): push into
                // the interior, slacks = d(x) pushed, bound multipliers = 1, zero step
                if (isS) push_interior(L.sv, c.vLo, c.vHi);
                if (isU) { push_interior(L.ua, c.aLo, c.aHi); push_interior(L.ud, c.dLo, c.dHi); }
                double prv[2];
                { const double u[2] = {L.ua, L.ud}; xprev<2>(u, prv); }
                const double pa = prv[0], pd = prv[1];
                if (isR) {
                    const double h0 = rHi(0), h1 = rHi(1);
                    L.rs[0] = L.ud - ((k == 0) ? cst(4) : pd);
                    L.rs[1] = L.ua - ((k == 0) ? cst(5) : pa);
                    push_interior(L.rs[0], -h0, h0); push_interior(L.rs[1], -h1, h1);
                }
                BoundMult Z;
                Z.zvL = Z.zvU = isS ? 1.0 : 0.0;
                Z.zaL = Z.zaU = Z.zdL = Z.zdU = isU ? 1.0 : 0.0;
                Z.rvL[0] = Z.rvL[1] = Z.rvU[0] = Z.rvU[1] = isR ? 1.0 : 0.0;
                st_z(Z);
                StepState D;
                D.dsx = D.dsy = D.dsp = D.dsv = D.dua = D.dud = 0.0; D.drs[0] = D.drs[1] = 0.0;
                D.nyx = D.nyy = D.nyp = D.nyv = 0.0; D.nyd[0] = D.nyd[1] = 0.0;
                st_dx(D); st_drs(D); st_dy(D);
                phase = PH_EVAL0; do_eval = true; ev_alpha = 0.0;
                continue;
            }
            if (phase == PH_EVAL0) {
                if (resto_check) {   // the restored point must be acceptable to the filter
                    const double th_r = ev.theta, ph_r = sigma * ev.f - mu * ev.lb;
                    bool ok = (th_r == th_r) && (ph_r == ph_r) && cmp_le(th_r, theta_max, theta_max);
                    const bool mine = (k >= nfilt) || cmp_le(ph_r, f_phi, f_phi) || cmp_le(th_r, f_theta, f_theta);
                    ok = tall(mine) && ok;
                    if (!ok) { ret = -2; break; }
                    resto_check = false;
                }
                cur_theta = ev.theta; cur_f = ev.f; cur_lb = ev.lb;
                phase = PH_LS; do_solve = true; req = 0;
                continue;
            }
            if (phase == PH_LS) {
                bool use = solve_ok;
                StepState D;
                ld_dy(D);
                if (solve_ok) {
                    double ym = dmax_(dmax_(fabs(D.nyx), fabs(D.nyy)), dmax_(fabs(D.nyp), fabs(D.nyv)));
                    ym = dmax_(ym, dmax_(fabs(D.nyd[0]), fabs(D.nyd[1])));
                    ym = tmax(isS ? ym : 0.0);
                    use = (ym <= K_Y_INIT_MAX);
                }
                if (use && isS) { L.yx = D.nyx; L.yy = D.nyy; L.yp = D.nyp; L.yv = D.nyv; L.ryd[0] = D.nyd[0]; L.ryd[1] = D.nyd[1]; }
                phase = PH_BEGIN;
            }
            if (phase == PH_BEGIN) {
                const Grad g = objective_gradient();
                const double gx = g.x, gy = g.y, gp = g.p, gv = g.v, ga = g.a, gd = g.d;
                EvalLane e;
                ev_load_model(e);
                ev_load_resid(e);
                BoundMult Z;
                ld_z(Z);
                const double A02 = isU ? -c.dt * L.sv * e.sn : 0.0, A03 = isU ? c.dt * e.cs : 0.0;
                const double A12 = isU ? c.dt * L.sv * e.cs : 0.0, A13 = isU ? c.dt * e.sn : 0.0;
                const double A23 = isU ? c.dtLb * e.sb : 0.0;
                const double b0 = A02 * e.b1, b1v = A12 * e.b1, b2v = isU ? c.dtLb * L.sv * e.cb * e.b1 : 0.0;
                double di, cv, cm0, cmm, sumy, sumz;
                {
                    double y1[6];
                    { const double y[6] = {L.yx, L.yy, L.yp, L.yv, L.ryd[0], L.ryd[1]}; xnext<6>(y, y1); }
                    const double y1x = y1[0], y1y = y1[1], y1p = y1[2], y1v = y1[3], yd1_0 = y1[4], yd1_1 = y1[5];
                    const double hn = isU ? 1.0 : 0.0;
                    double glx = gx + L.yx - hn * y1x;
                    double gly = gy + L.yy - hn * y1y;
                    double glp = gp + L.yp - hn * (A02 * y1x + A12 * y1y + y1p);
                    double glv = gv + L.yv - hn * (A03 * y1x + A13 * y1y + A23 * y1p + y1v) - Z.zvL + Z.zvU;
                    double jd = b0 * y1x + b1v * y1y + b2v * y1p;
                    if (MODEL) {
                        const FJac J = frenet_jac(e);
                        glx = gx + L.yx - (J.a00 * y1x + J.a20 * y1p);
                        gly = gy + L.yy - (J.a01 * y1x + hn * y1y + J.a21 * y1p);
                        glp = gp + L.yp - (J.a02 * y1x + J.a12 * y1y + J.a22 * y1p);
                        glv = gv + L.yv - (J.a03 * y1x + J.a13 * y1y + J.a23 * y1p + hn * y1v) - Z.zvL + Z.zvU;
                        jd = J.b0 * y1x + J.b1 * y1y + J.b2 * y1p;
                    }
                    const double nd0 = (k + 1 < N) ? yd1_0 : 0.0, nd1 = (k + 1 < N) ? yd1_1 : 0.0;
                    const double gla = ga - hn * c.dt * y1v + (L.ryd[1] - nd1) - Z.zaL + Z.zaU;
                    const double gld = gd - hn * jd + (L.ryd[0] - nd0) - Z.zdL + Z.zdU;
                    di = dmax_(dmax_(fabs(glx), fabs(gly)), dmax_(fabs(glp), fabs(glv)));
                    di = dmax_(di, dmax_(fabs(gla), fabs(gld)));
                    di = dmax_(di, dmax_(fabs(-L.ryd[0] - Z.rvL[0] + Z.rvU[0]), fabs(-L.ryd[1] - Z.rvL[1] + Z.rvU[1])));
                    di = isS ? di : 0.0;
                    cv = dmax_(dmax_(fabs(e.rd[0]), fabs(e.rd[1])), dmax_(fabs(e.rd[2]), fabs(e.rd[3])));
                    cv = dmax_(cv, dmax_(fabs(e.dr[0]), fabs(e.dr[1])));
                    sumy = isS ? fabs(L.yx) + fabs(L.yy) + fabs(L.yp) + fabs(L.yv) + fabs(L.ryd[0]) + fabs(L.ryd[1]) : 0.0;
                    sumz = Z.zvL + Z.zvU + Z.zaL + Z.zaU + Z.zdL + Z.zdU + Z.rvL[0] + Z.rvL[1] + Z.rvU[0] + Z.rvU[1];
                    double r2[2] = {sumy, sumz};
                    treduce<OP_SUM, 2>(r2);
                    sumy = r2[0]; sumz = r2[1];
                }
                // s_d, s_c = max(s_max, mean |multiplier|) / s_max: exactly 1 unless the multipliers are huge
                const double sty = sumy + sumz;
                const bool big_d = sty > K_S_MAX * (double)(my + nz), big_c = sumz > K_S_MAX * (double)nz;
                double sd = 1.0, sc = 1.0;
                if (big_d) sd = div_cold(sty, (double)(my + nz) * K_S_MAX);
                if (big_c) sc = div_cold(sumz, (double)nz * K_S_MAX);
                // complementarity of this lane: max |slack * z - t| over its bound pairs
                // (the ten slack * z products once; pairs this thread does not own repeat its v pair,
                // which every stage thread owns, so that they do not change the maximum)
                double pz[10];
                pz[0] = (L.sv - c.vLo) * Z.zvL; pz[1] = (c.vHi - L.sv) * Z.zvU;
                pz[2] = isU ? (L.ua - c.aLo) * Z.zaL : pz[0]; pz[3] = isU ? (c.aHi - L.ua) * Z.zaU : pz[0];
                pz[4] = isU ? (L.ud - c.dLo) * Z.zdL : pz[0]; pz[5] = isU ? (c.dHi - L.ud) * Z.zdU : pz[0];
                {
                    const double h0 = rHi(0), h1 = rHi(1);
                    pz[6] = isR ? (L.rs[0] + h0) * Z.rvL[0] : pz[0]; pz[7] = isR ? (h0 - L.rs[0]) * Z.rvU[0] : pz[0];
                    pz[8] = isR ? (L.rs[1] + h1) * Z.rvL[1] : pz[0]; pz[9] = isR ? (h1 - L.rs[1]) * Z.rvU[1] : pz[0];
                }
                auto compl_local = [&](double t) {
                    double m = 0.0;
                    for (int i = 0; i < 10; i++) m = dmax_(m, fabs(pz[i] - t));
                    return isS ? m : 0.0;
                };
                cm0 = compl_local(0.0); cmm = compl_local(mu);
                // E_0 and E_mu in one pass
                const double dcv = dmax_(big_d ? div_cold(di, sd) : di, cv);
                double e0, em;
                {
                    double r2[2] = {dmax_(dcv, big_c ? div_cold(cm0, sc) : cm0), dmax_(dcv, big_c ? div_cold(cmm, sc) : cmm)};
                    treduce<OP_MAX, 2>(r2);
                    e0 = r2[0]; em = r2[1];
                }
#ifdef MPC_TRACE
                if (k == 0) printf("it %3d mu %.2e e0 %.3e em %.3e theta %.2e f %.10e dcv %.2e cm0 %.2e nfilt %d\n", iter, mu, e0, em, cur_theta, cur_f, dcv, cm0, nfilt);
#endif
                // ---- convergence (OptimalityErrorConvergenceCheck)
                if (e0 <= dmax_(K_ACCEPT_TOL, c.tol)) {   // the unscaled checks need three more reductions: only near the end
                    double r3[3] = {di, cv, cm0};
                    treduce<OP_MAX, 3>(r3);
                    const double du = r3[0] / sigma, cvm = r3[1], mc = r3[2] / sigma;
                    if (e0 <= c.tol && du <= 1.0 && cvm <= 1e-4 && mc <= 1e-4) { ret = 0; break; }
                    cur_acceptable = (e0 <= K_ACCEPT_TOL && du <= 1e10 && cvm <= 1e-2 && mc <= 1e-2);
                    if (cur_acceptable) { had_acceptable = true; if (++accept_count >= K_ACCEPT_ITER) { ret = 1; break; } }
                    else accept_count = 0;
                } else { accept_count = 0; cur_acceptable = false; }
                if (iter >= c.max_iter) { ret = -1; break; }
                {
                    const double xm = dmax_(dmax_(fabs(L.sx), fabs(L.sy)), dmax_(fabs(L.sp), fabs(L.sv)));
                    if (!tall(!isS || xm <= 1e20)) { ret = -5; break; }
                }
                // ---- monotone barrier update
                for (;;) {
                    if (!(em <= K_KAPPA_EPS * mu) && !tiny_last) break;
                    const double nm = dmax_(c.mu_min, dmin_(K_KAPPA_MU * mu, mu * sqrt(mu)));
                    if (nm >= mu) { if (tiny_last) ret = -3; break; }
                    mu = nm; tau = dmax_(K_TAU_MIN, 1.0 - mu);
                    nfilt = 0;
                    if (tiny_last) { tiny_last = false; break; }
                    const double cl = compl_local(mu);
                    em = tmax(dmax_(dcv, big_c ? div_cold(cl, sc) : cl));
                }
                if (ret == -3) break;
                dw = 0.0;
                phase = PH_PD; do_solve = true; req = 1;
                continue;
            }
            if (phase == PH_RESOLVE_EVAL) {
                phase = PH_RESOLVE; do_solve = true; req = 1;
                continue;
            }
            if (phase == PH_PD || phase == PH_RESOLVE) {
                if (!solve_ok) {
                    // PDPerturbationHandler::PerturbForWrongInertia
                    if (dw == 0.0) dw = (dw_last == 0.0) ? K_DW_INIT : dmax_(K_DW_MIN, dw_last * K_DW_DEC);
                    else dw = (dw_last == 0.0 || 1e5 * dw_last < dw) ? K_DW_INC_FIRST * dw : K_DW_INC * dw;
                    if (dw > K_DW_MAX) { ret = -4; break; }
                    do_solve = true; req = 2;
                    continue;
                }
                if (phase == PH_RESOLVE) {
                    alpha = alpha_max * 0.5; nsteps = 1;
                    double alpha_min = K_GAMMA_THETA;
                    if (gBd < 0.0) alpha_min = dmin_(K_GAMMA_THETA, K_GAMMA_PHI * cur_theta / (-gBd));
                    bool above_min = alpha > alpha_min * K_ALPHA_MIN_FRAC;
                    if (!above_min && gBd < 0.0 && cur_theta <= theta_min)
                        above_min = ratio_test(1, alpha, K_ALPHA_MIN_FRAC * (K_DELTA * Rft), cur_theta, -gBd);
                    if (!above_min) {
                        if (cur_acceptable) { ret = 1; break; }
                        if (cur_theta <= 1e-2 * c.tol) { ret = had_acceptable ? 1 : -2; break; }
                        if (n_resto < K_MAX_RESTO) { phase = PH_RESTO; continue; }
                        ret = -2; break;
                    }
                    ev_alpha = alpha; do_eval = true; phase = PH_TRIAL;
                    continue;
                }
                if (dw > 0.0) dw_last = dw;
                // ---- line-search quantities at the current point
                const double theta = cur_theta;
                phi = sigma * cur_f - mu * cur_lb;
                {
                    // grad(phi)'d from the condensed gradient in the record:
                    //   sum g~ dx + sum_rows [ br rdr - SrW rdr (drs - rdr) ]
                    const int r = rec();
                    StepState D;
                    ld_dx(D); ld_drs(D);
                    double t = 0.0;
                    bool tl = true;  // all |dx_i| < 10 eps (1 + |x_i|)
                    const double tt = 10.0 * K_EPS;
                    if (isS) {
                        const d2 g01 = lds2(sm, r + SO(SD_GX)), g23 = lds2(sm, r + SO(SD_GX + 2)), g45 = lds2(sm, r + SO(SD_GX + 4));
                        t = g01.x * D.dsx + g01.y * D.dsy + g23.x * D.dsp + g23.y * D.dsv + g45.x * D.dua + g45.y * D.dud;
                        tl = fabs(D.dsx) < tt * (1.0 + fabs(L.sx)) && fabs(D.dsy) < tt * (1.0 + fabs(L.sy)) &&
                             fabs(D.dsp) < tt * (1.0 + fabs(L.sp)) && fabs(D.dsv) < tt * (1.0 + fabs(L.sv)) &&
                             fabs(D.dua) < tt * (1.0 + fabs(L.ua)) && fabs(D.dud) < tt * (1.0 + fabs(L.ud)) &&
                             fabs(D.drs[0]) < tt * (1.0 + fabs(L.rs[0])) && fabs(D.drs[1]) < tt * (1.0 + fabs(L.rs[1]));
                    }
                    if (isR) {
                        const d2 srw = lds2(sm, r + SO(SD_SRW)), brr = lds2(sm, r + SO(SD_BR)), drr = lds2(sm, r + SO(SD_DR));
                        t += brr.x * drr.x - srw.x * drr.x * (D.drs[0] - drr.x);
                        t += brr.y * drr.y - srw.y * drr.y * (D.drs[1] - drr.y);
                    }
                    gBd = tsum(t);
                    tiny = tall(tl) && (theta < 1e-4);
                }
                if (theta_max < 0.0) { theta_max = 1e4 * dmax_(1.0, theta); theta_min = 1e-4 * dmax_(1.0, theta); }
                // switching-condition ratio theta^s_theta / (-gBd)^s_phi, single-precision estimate (see ratio_test)
                Rft = (gBd < 0.0) ? (double)fast_exp2((float)K_S_THETA * fast_log2((float)theta) - (float)K_S_PHI * fast_log2((float)(-gBd))) : 0.0;
                alpha_max = alpha_primal(tau);
                alpha = alpha_max; nsteps = 0;
                ev_alpha = alpha; do_eval = true; phase = PH_TRIAL;
                continue;
            }
        }
        res.iters = iter; res.n_resto = n_resto;
        res.status = (ret == 0 || ret == 1) ? 0 : (ret == 2 ? 1 : (ret == -1 ? 3 : (ret == -5 ? 2 : 4)));
        // honor_original_bounds
        if (feasible) {
            if (isS) L.sv = dmin_(dmax_(L.sv, c.vmin), c.vmax);
            if (isU) { L.ua = dmin_(dmax_(L.ua, -c.amax), c.amax); L.ud = dmin_(dmax_(L.ud, -c.smax), c.smax); }
        }
        {   // unscaled objective at the returned point
            double prv[2];
            { const double u[2] = {L.ua, L.ud}; xprev<2>(u, prv); }
            const double pa = prv[0], pd = prv[1];
            const double ex = L.sx - ref_x(), ey = L.sy - ref_y(), ep = L.sp - ref_p(), evv = L.sv - cst(6);
            double f = wx() * ex * ex + wy() * ey * ey + wp() * ep * ep + wv() * evv * evv;
            if (isU) {
                f += wt(6) * L.ua * L.ua + wt(7) * L.ud * L.ud;
                if (k >= 1) { const double da = L.ua - pa, dd = L.ud - pd; f += wt(4) * da * da + wt(5) * dd * dd; }
            }
            res.cost = tsum(f);
        }
        return res;
    }
};

// Problem I/O for one warp: problem-major layouts of include/mpc_b200.h.
struct BatchPtrs {
    const double* state;   // [B][4]
    const double* ref;     // [B][3][N+1]
    const double* v_des;   // [B] or null
    const double* u_prev;  // [B][2]
    double* warm;          // [B][6N+4] or null
    double* u0;            // [B][2] or null (when rec is given)
    double* cost;          // [B] or null
    int* status;           // [B] or null
    int* iters;            // [B] or null
    double* traj;          // [B][6N+4] or null
    double* rec;           // [B][4] or null: the packed 32-byte result record {acc, df, cost: f64; status, iters: i32} that the
                           //   multi-GPU all-gather moves (SURVEY 8e); its status word carries the restoration count in bits 8..15
    int* resto;            // [B] or null: restorations by rollout this solve went through (0 for almost every problem)
    const double* w;       // [B][8] ([B][7] Frenet) or null: the problem's own cost weights (row_weight); null = KCfg::w
};

// The answer to a problem that cannot be solved as given (a path id never set, a weight row that is negative or NaN -- device
// pointers cannot be checked on the host): MPCB200_ERROR, zero commands, cost 0, no iterations, no restorations
MPC_DEV void write_error_answer(const BatchPtrs& io, long b) {
    if (io.u0) { io.u0[2 * b] = 0.0; io.u0[2 * b + 1] = 0.0; }
    if (io.cost) io.cost[b] = 0.0;
    if (io.status) io.status[b] = 4;
    if (io.iters) io.iters[b] = 0;
    if (io.rec) { st_global_v2(io.rec + 4 * b, 0.0, 0.0); st_global_v2(io.rec + 4 * b + 2, 0.0, int2_as_double(4, 0)); }
    if (io.resto) io.resto[b] = 0;
}

// Optional on-device reference generation for a batch (path_of != null): the waypoints come from the
// replicated path tables instead of io.ref.
struct RefGen {
    const int* path_of;     // [B] index into paths[], or null: references are read from io.ref
    PathTable paths[3];
    int track_using_time;
    double target_vel;      // arc-length spacing of the waypoints when !track_using_time
    double* ref_out;        // [B][3][N+1] or null: the generated waypoints (target_path of mpc_cmd_pub.jl:134-138)
    int* stop;              // [B] or null: stop_cmd of get_waypoints
};

// MODEL 1 (Frenet-frame variant): io.state = (s, e_y, e_psi, v), io.ref = [B][4] curvature polynomial (highest degree
// first), traj / warm = s, e_y, v, e_psi, d_f, acc (get_solver_results of MKZMPCPathFollowerFrenet.jl:188-206)
// PW: the problem's weights come from io.w (KCfg::w when it is null); a row that breaks mpcb200_set_cost's rule gets
// write_error_answer
template <int W, int MODEL = 0, int PW = 0>
MPC_DEV void solve_problem(const KCfg& cfg, const BatchPtrs& io, const RefGen& rg, long b, smem_t smem) {
    TeamSolver<W, MODEL, PW> S(cfg, smem);
    const int k = S.k, N = cfg.N;
    const long nr = 3L * (N + 1), nt = 6L * N + 4;
    if (MODEL) {
        const double* kp = io.ref + 4 * b;
        S.set_kpoly(kp[0], kp[1], kp[2], kp[3]);
    } else if (rg.path_of) {
        // ---- waypoints from the path table: nearest sample to (X, Y), then interpolation and heading unwrap
        const int pid = rg.path_of[b];
        if (pid < 0 || pid > 2 || rg.paths[pid].n < 2) {
            // a path id that was never given to mpcb200_set_path (device pointers cannot be checked on the host):
            // the problem is answered with MPCB200_ERROR and zero commands instead of indexing outside the tables
            if (k == 0) {
                write_error_answer(io, b);
                if (rg.stop) rg.stop[b] = 0;
            }
            return;
        }
        double xr, yr, pr;
        const bool sc = S.get_waypoints(rg.paths[pid], cfg.dt, io.state[4 * b], io.state[4 * b + 1], io.state[4 * b + 2],
                                        !rg.track_using_time, rg.target_vel, xr, yr, pr);
        S.set_ref(xr, yr, pr);
        if (rg.ref_out && k <= N) { double* ro = rg.ref_out + nr * b; ro[k] = xr; ro[(N + 1) + k] = yr; ro[2 * (N + 1) + k] = pr; }
        if (rg.stop && k == 0) rg.stop[b] = sc ? 1 : 0;
    } else {
        // ---- coalesced loads: lane k takes stage k's reference sample
        const double* rf = io.ref + nr * b;
        S.set_ref((k <= N) ? rf[k] : 0.0, (k <= N) ? rf[(N + 1) + k] : 0.0, (k <= N) ? rf[2 * (N + 1) + k] : 0.0);
    }
    {   // lanes 0..6: the problem constants
        double cv = 0.0;
        if (k < 4) cv = io.state[4 * b + k];
        else if (k < 6) cv = io.u_prev[2 * b + (k - 4)];
        else if (k == 6) cv = io.v_des ? io.v_des[b] : (rg.path_of ? rg.target_vel : 0.0);   // des_speed (clamped on the host), mpc_cmd_pub.jl:58-62,116
        if (k < 8) sts(smem, SO(W_CONST + k), cv);
        if (PW) {
            const double wk = (k < 8) ? (io.w ? row_weight(io.w, b, k, MODEL) : cfg.w[k]) : 0.0;
            if (k < 8) sts(smem, SO(wt_offset(N, MODEL) + k), wk);
            if (!S.tall(wk >= 0.0)) {
                if (k == 0) write_error_answer(io, b);
                S.tsync();
                return;
            }
        }
        S.tsync();
    }
    // ---- start point
    S.L.sx = S.L.sy = S.L.sp = S.L.sv = S.L.ua = S.L.ud = 0.0;
    if (io.warm) {
        const double* w = io.warm + nt * b;
        if (k <= N) { S.L.sx = w[k]; S.L.sy = w[(N + 1) + k]; S.L.sv = w[2 * (N + 1) + k]; S.L.sp = w[3 * (N + 1) + k]; }
        if (k < N) { S.L.ud = w[4 * (N + 1) + k]; S.L.ua = w[4 * (N + 1) + N + k]; }
    } else if (cfg.start_mode == 1) {
        // MPCB200_START_ROLLOUT (opt-in, not a reference behaviour): hold the previous command over the
        // horizon (projected onto the box and rate rows) and roll the model out from the measured state
        if (k < N) { S.L.ua = S.cst(5); S.L.ud = S.cst(4); }
        S.rollout_restore();
    }
    const Result r = S.solve();
    // ---- results
    const double a0 = S.bcast0(S.L.ua), d0 = S.bcast0(S.L.ud);
    if (k == 0) {
        if (io.u0) { io.u0[2 * b] = a0; io.u0[2 * b + 1] = d0; }
        if (io.cost) io.cost[b] = r.cost;
        if (io.status) io.status[b] = r.status;
        if (io.iters) io.iters[b] = r.iters;
        if (io.rec) { st_global_v2(io.rec + 4 * b, a0, d0); st_global_v2(io.rec + 4 * b + 2, r.cost, int2_as_double(r.status | (r.n_resto << 8), r.iters)); }
        if (io.resto) io.resto[b] = r.n_resto;
    }
    for (int pass = 0; pass < 2; pass++) {
        double* t = (pass == 0) ? io.traj : io.warm;
        if (!t) continue;
        t += nt * b;
        if (k <= N) { t[k] = S.L.sx; t[(N + 1) + k] = S.L.sy; t[2 * (N + 1) + k] = S.L.sv; t[3 * (N + 1) + k] = S.L.sp; }
        if (k < N) { t[4 * (N + 1) + k] = S.L.ud; t[4 * (N + 1) + N + k] = S.L.ua; }
    }
    S.tsync();
}


// ======================================================================================
// Closed-loop rollout: one warp = one vehicle for T control steps, everything on the device.
//   plant              scripts/vehicle_simulator.py:58-112  (10 publishes x 10 Euler sub-steps per control period)
//   reference          scripts/gps_utils/ref_gps_traj.py:131-218 (nearest sample, np.interp, heading unwrap, stop_cmd)
//   control step       scripts/mpc_cmd_pub.jl:86-157 (warm-started solve, command fed back, stop latch)
// ======================================================================================
struct RolloutArgs {
    const double* pose0;    // [B][3] X0, Y0, Psi0
    const int* path_of;     // [B] index into paths[]
    PathTable paths[3];
    int T, track_using_time;
    double target_vel;
    double* log;            // [T][B][8] or null
    double* final_state;    // [B][8] or null
    long B;
    const double* warm0;    // [6N+4] or null: start point of every vehicle's FIRST solve (the module-load solution)
    const double* w;        // [B][8] or null: each vehicle's cost weights for all its control periods (checked by the host); null = KCfg::w
};

// atan2(y, x) for x > 0 and sincos for small arguments: the plant's slip angles and steering angle are
// small, where a short Taylor sum is accurate to the last bits (truncation < 1e-21 for |y/x| <= 1/8 and
// < 1e-24 for |x| <= 0.6) and several times shorter than the general routines, which stay as fall-back
MPC_DEV double atan2_posx(double y, double x) {
    const double t = y / x;
    if (!(fabs(t) <= 0.125)) return atan2(y, x);
    const double u = t * t;
    double p = 1.0 / 21.0;
    p = 1.0 / 19.0 - u * p; p = 1.0 / 17.0 - u * p; p = 1.0 / 15.0 - u * p; p = 1.0 / 13.0 - u * p; p = 1.0 / 11.0 - u * p;
    p = 1.0 / 9.0 - u * p; p = 1.0 / 7.0 - u * p; p = 1.0 / 5.0 - u * p; p = 1.0 / 3.0 - u * p; p = 1.0 - u * p;
    return t * p;
}
MPC_DEV void sincos_small(double x, double* s, double* c) {
    if (!(fabs(x) <= 0.6)) { mpc_sincos(x, s, c); return; }
    const double u = x * x;
    double ps = -1.0 / 6.0 + u * (1.0 / 120.0 + u * (-1.0 / 5040.0 + u * (1.0 / 362880.0 + u * (-1.0 / 39916800.0 + u * (1.0 / 6227020800.0 +
                u * (-1.0 / 1307674368000.0 + u * (1.0 / 355687428096000.0 + u * (-1.0 / 121645100408832000.0))))))));
    double pc = -0.5 + u * (1.0 / 24.0 + u * (-1.0 / 720.0 + u * (1.0 / 40320.0 + u * (-1.0 / 3628800.0 + u * (1.0 / 479001600.0 +
                u * (-1.0 / 87178291200.0 + u * (1.0 / 20922789888000.0 + u * (-1.0 / 6402373705728000.0 + u * (1.0 / 2432902008176640000.0)))))))));
    *s = x + x * (u * ps);
    *c = 1.0 + u * pc;
}

MPC_DEV double py_mod(double a, double m) { double r = fmod(a, m); if (r != 0.0 && ((r < 0.0) != (m < 0.0))) r += m; return r; }

// vehicle_simulator.py:58-112, one 100 Hz publish period; st = X,Y,psi,vx,vy,wz,acc,df (every lane computes the same)
MPC_DEV void plant_step(double* st, double acc_des, double df_des) {
    const double lf = 1.152, lr = 1.693, m = 1840.0, Iz = 3477.0, Caf = 4.0703e4, Car = 6.4495e4;
    const double deltaT = 0.01 / 10.0, PI = 3.141592653589793;
    for (int i = 0; i < 10; i++) {
        const double X = st[0], Y = st[1], psi = st[2], vx = st[3], vy = st[4], wz = st[5], acc = st[6], df = st[7];
        double af = 0.0, ar = 0.0;
        if (vx > 1e-6) { af = df - atan2_posx(vy + lf * wz, vx); ar = -atan2_posx(vy - lf * wz, vx); }   // :77 uses lf (sic); vx >= 0 (clamped below)
        const double Fyf = Caf * af, Fyr = Car * ar;
        double sdf, cdf, sps, cps;
        sincos_small(df, &sdf, &cdf);
        mpc_sincos(psi, &sps, &cps);
        // :86 `1/m*Fyf*np.sin(self.df)`: the node is Python 2 and m an int, so 1/m == 0 and the term is (+-)0
        double vx_n = vx + deltaT * (acc - 0.0 * Fyf * sdf + wz * vy);
        if (vx_n < 0.0) vx_n = 0.0;
        double vy_n = 0.0, wz_n = 0.0;
        if (vx_n > 1e-6) {
            vy_n = vy + deltaT * (1.0 / m * (Fyf * cdf + Fyr) - wz * vx);
            wz_n = wz + deltaT * (1.0 / Iz * (lf * Fyf * cdf - lr * Fyr));
        }
        const double psi_n = psi + deltaT * wz;
        st[0] = X + deltaT * (vx * cps - vy * sps);
        st[1] = Y + deltaT * (vx * sps + vy * cps);
        const double pw = psi_n + PI;   // np.mod(a, m) is a itself for 0 <= a < m: fmod only when the yaw really wraps
        st[2] = ((pw >= 0.0 && pw < 2.0 * PI) ? pw : py_mod(pw, 2.0 * PI)) - PI;
        st[3] = vx_n; st[4] = vy_n; st[5] = wz_n;
        st[6] = 5.0 * (acc_des - acc) * deltaT + acc;
        st[7] = 5.0 * (df_des - df) * deltaT + df;
    }
}

MPC_DEV double sel8(const double* v, int i) {   // register-friendly v[i] for a lane-dependent i
    return (i == 0) ? v[0] : (i == 1) ? v[1] : (i == 2) ? v[2] : (i == 3) ? v[3] : (i == 4) ? v[4] : (i == 5) ? v[5] : (i == 6) ? v[6] : v[7];
}

// One block = `nwarps` vehicles (one per warp, W = 1) stepping through the T control periods together, or ONE vehicle
// whose problem is shared by the W = 2, 3 warps of the block (long horizons).
// The plant of all the block's vehicles is integrated by ONE warp, lane = vehicle (every lane of a
// warp would otherwise repeat the same 100 Euler sub-steps, atan2 and sincos included: 40 % of the
// rollout's instructions); states and commands cross through `px` ([vehicle][10] doubles) around two
// block barriers per control period.  Warps whose vehicle index is past the fleet only keep the barriers.
#define ROLLOUT_PX 10   // X, Y, psi, vx, vy, wz, acc, df, acc_des, df_des
template <int W, int PW = 0>
MPC_DEV void rollout_group(const KCfg& cfg, const RolloutArgs& a, long b0, smem_t smem, smem_t px, int nwarps) {
    TeamSolver<W, 0, PW> S(cfg, smem);
    const int k = S.k, N = cfg.N;
    const int w = (W == 1) ? (thread_in_block() >> 5) : 0;   // vehicle of this thread within the block
    const int nveh = (W == 1) ? nwarps : 1;
    const long b = b0 + w;
    const bool valid = b < a.B;
    const int pxw = SO(w * ROLLOUT_PX);
    const PathTable& path = a.paths[valid ? a.path_of[b] : 0];
    if (k < 8) sts(px, pxw + SO(k), (valid && k < 3) ? a.pose0[3 * b + k] : 0.0);
    if (PW && k < 8) sts(smem, SO(wt_offset(N, 0) + k), (valid && a.w) ? a.w[8 * b + k] : cfg.w[k]);   // the vehicle keeps its row
    double st[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    double acc_des = 0.0, df_des = 0.0, up_d = 0.0, up_a = 0.0;   // commands, d_f_current, acc_current
    const double des_speed = a.target_vel > 0.0 ? a.target_vel : 0.0;
    bool stop = false;
    // the first solve of the node starts from the solution of the module-load solve of the default problem
    // (MKZMPCPathFollower.jl:126-128: JuMP re-solves from the previous primal values); later ones from the previous solution
    S.L.sx = S.L.sy = S.L.sp = S.L.sv = S.L.ua = S.L.ud = 0.0;
    if (a.warm0) {
        const double* w0 = a.warm0;
        if (k <= N) { S.L.sx = w0[k]; S.L.sy = w0[(N + 1) + k]; S.L.sv = w0[2 * (N + 1) + k]; S.L.sp = w0[3 * (N + 1) + k]; }
        if (k < N) { S.L.ud = w0[4 * (N + 1) + k]; S.L.ua = w0[4 * (N + 1) + N + k]; }
    }
    for (int t = 0; t < a.T; t++) {
        if (k == 0) { sts(px, pxw + SO(8), acc_des); sts(px, pxw + SO(9), df_des); }
        block_sync();
        if (thread_in_block() < nveh) {   // lane = vehicle: ten 100 Hz publishes of ten Euler sub-steps each
            const int pv = SO(thread_in_block() * ROLLOUT_PX);
            double ps[8];
            for (int i = 0; i < 8; i++) ps[i] = lds(px, pv + SO(i));
            const double ad = lds(px, pv + SO(8)), dd = lds(px, pv + SO(9));
            MPC_NOUNROLL for (int i = 0; i < 10; i++) plant_step(ps, ad, dd);
            for (int i = 0; i < 8; i++) sts(px, pv + SO(i), ps[i]);
        }
        block_sync();
        if (!valid) continue;
        for (int i = 0; i < 8; i++) st[i] = lds(px, pxw + SO(i));
        double xr, yr, pr;
        const bool sc = S.get_waypoints(path, cfg.dt, st[0], st[1], st[2], !a.track_using_time, des_speed, xr, yr, pr);
        S.set_ref(xr, yr, pr);
        if (sc) stop = true;   // latch, mpc_cmd_pub.jl:102-111
        int status = -1, iters = 0;
        if (!stop) {
            S.tsync();
            {
                const double cv[8] = {st[0], st[1], st[2], st[3], up_d, up_a, des_speed, 0.0};
                if (k < 8) sts(smem, SO(W_CONST + k), sel8(cv, k));
            }
            S.tsync();
            const Result r = S.solve();
            status = r.status; iters = r.iters;
            acc_des = S.bcast0(S.L.ua); df_des = S.bcast0(S.L.ud);   // published whatever the status (:129-132)
            up_d = df_des; up_a = acc_des;                           // update_current_input(df_opt, a_opt) (:140)
        } else { acc_des = -1.0; df_des = 0.0; }                     // :148-153
        if (a.log && k < 8) {
            const double lv[8] = {st[0], st[1], st[2], st[3], acc_des, df_des, (double)status, (double)iters};
            a.log[((long)t * a.B + b) * 8 + k] = sel8(lv, k);
        }
    }
    if (valid && a.final_state && k < 8) a.final_state[b * 8 + k] = sel8(st, k);
    block_sync();
}


// ======================================================================================
// Closed loop on the Frenet-frame module, everything on the device: one warp = one vehicle.
//   control step       scripts/nodes_gazebo_sim/gazebo_sim_mpc_cmd_pub_frenet.jl:112-153 (state (0, e_y, -psi_start, v),
//                      K_coeffs from the path ahead, warm-started solve, command fed back)
//   curvature fit      scripts/sim_path_utils/nav_msgs_path_frenet.py:44-86: cubics X(s), Y(s) fitted to the path ahead
//                      resampled every 0.5 m (:60-72), curvature of those cubics every 0.25 m fitted by a cubic (:44-58),
//                      psi_start = atan2(Y'(0), X'(0)) (:84).  Both least-squares fits are on FIXED grids, so each is one
//                      fixed 4 x n matrix (the pseudo-inverse of the Vandermonde matrix, built once by the host) times the
//                      samples: lanes stride the samples, the 4 + 4 + 4 partial sums are reduced over the warp.
//   path ahead         the next `window` metres of the recorded path from the sample nearest to the vehicle, seen from the
//                      vehicle (what the node receives as `target_path`, :90-119), as closed_loop.run_frenet builds it
//   plant              scripts/vehicle_simulator.py:58-112 (Gazebo, which drives that node in the reference, is out of scope)
// ======================================================================================
struct FrenetRolloutArgs {
    const double* pose0;    // [B][3] X0, Y0, Psi0
    const int* path_of;     // [B]
    PathTable paths[3];
    int T, ey_from_path;
    double target_vel;
    double* log;            // [T][B][8] or null: x, y, psi, v, acc_cmd, df_cmd, status, iters
    double* final_state;    // [B][8] or null
    long B;
    const double* P1;       // [4][n1] least-squares cubic fit on the grid 0, 0.5, ... (n1 samples)
    const double* P2;       // [4][n2] ... on the grid 0, 0.25, ... (n2 samples)
    int n1, n2;
};

// host side: the fit matrices of FrenetRolloutArgs
// Sizes of the two fit grids, those of nav_msgs_path_frenet.py:63,79: np.arange(0, window, 0.5) and np.arange(0, window, 0.25)
// have ceil(window / step) samples.  Dividing by 0.5 or 0.25 is exact, so no tolerance is needed (one would drop a sample of
// a window just above a multiple of the step).
inline void fit_grid_sizes(double window, int* n1, int* n2) {
    *n1 = (int)ceil(window / 0.5);
    *n2 = (int)ceil(window / 0.25);
}
// Least-squares cubic fit on the fixed grid x_g = g * step, g < n, as a 4 x n matrix P (coefficients, highest degree first,
// = P * samples): P = (V'V)^-1 V' with the Vandermonde columns scaled to unit norm, normal equations in long double.
inline void cubic_fit_matrix(int n, double step, double* P) {
    long double scale[4], G[4][4], Ginv[4][8];
    for (int c = 0; c < 4; c++) {
        long double ss = 0;
        for (int g = 0; g < n; g++) { const long double x = (long double)step * g; long double v = 1; for (int e = 0; e < 3 - c; e++) v *= x; ss += v * v; }
        scale[c] = sqrtl(ss);
    }
    auto V = [&](int g, int c) { const long double x = (long double)step * g; long double v = 1; for (int e = 0; e < 3 - c; e++) v *= x; return v / scale[c]; };
    for (int a = 0; a < 4; a++) for (int b = 0; b < 4; b++) { long double t = 0; for (int g = 0; g < n; g++) t += V(g, a) * V(g, b); G[a][b] = t; }
    for (int a = 0; a < 4; a++) for (int b = 0; b < 8; b++) Ginv[a][b] = (b < 4) ? G[a][b] : (b - 4 == a ? 1.0L : 0.0L);
    for (int c = 0; c < 4; c++) {   /* Gauss-Jordan with partial pivoting on a 4 x 4 SPD matrix */
        int piv = c;
        for (int r = c + 1; r < 4; r++) if (fabsl(Ginv[r][c]) > fabsl(Ginv[piv][c])) piv = r;
        if (piv != c) for (int b = 0; b < 8; b++) { const long double t = Ginv[c][b]; Ginv[c][b] = Ginv[piv][b]; Ginv[piv][b] = t; }
        const long double d = Ginv[c][c];
        for (int b = 0; b < 8; b++) Ginv[c][b] /= d;
        for (int r = 0; r < 4; r++) if (r != c) { const long double f = Ginv[r][c]; for (int b = 0; b < 8; b++) Ginv[r][b] -= f * Ginv[c][b]; }
    }
    for (int a = 0; a < 4; a++)
        for (int g = 0; g < n; g++) { long double t = 0; for (int b = 0; b < 4; b++) t += Ginv[a][4 + b] * V(g, b); P[(size_t)a * n + g] = (double)(t / scale[a]); }
}


// The Frenet node's reference for one vehicle, computed by one warp (lane k): the path ahead of the nearest sample resampled every
// 0.5 m in the vehicle frame, X(s) and Y(s) fitted by cubics on that fixed grid (nav_msgs_path_frenet.py:60-72), the curvature of the
// fitted cubics every 0.25 m fitted by a cubic (:44-58), psi_start = atan2(Y'(0), X'(0)) (:84) and e_y.  Both least-squares fits are
// the host-built matrices P1, P2 times the samples: lanes stride the samples, the partial sums are reduced over the warp.  Used by
// the fused closed-loop kernel (rollout_group_frenet) and by the per-period pipeline (rollout_frenet_ref_kernel).
MPC_DEV void frenet_reference(TeamSolver<1, 1>& S, const PathTable& path, const FrenetRolloutArgs& a, double X, double Y, double yaw,
                              double kc[4], double& ey, double& psi0) {
    const int k = S.k;
    const int bi = S.nearest_sample(path, X, Y);
    const double s_i = path.s[bi];
    double sps, cps;
    mpc_sincos(yaw, &sps, &cps);
    double acc8[8] = {0, 0, 0, 0, 0, 0, 0, 0}, xw0 = 0.0, yw0 = 0.0;
    for (int g = k; g < a.n1; g += 32) {
        const double sq = s_i + 0.5 * (double)g;
        const double dx = np_interp(sq, path.s, path.X, path.n) - X, dy = np_interp(sq, path.s, path.Y, path.n) - Y;
        const double xw = cps * dx + sps * dy, yw = -sps * dx + cps * dy;
        if (g == 0) { xw0 = xw; yw0 = yw; }
        for (int r = 0; r < 4; r++) { const double pr = a.P1[r * a.n1 + g]; acc8[r] += pr * xw; acc8[4 + r] += pr * yw; }
    }
    S.template treduce<TeamSolver<1, 1>::OP_SUM, 3>(acc8); S.template treduce<TeamSolver<1, 1>::OP_SUM, 3>(acc8 + 3);
    S.template treduce<TeamSolver<1, 1>::OP_SUM, 2>(acc8 + 6);
    xw0 = shfl(xw0, 0); yw0 = shfl(yw0, 0);
    const double* xc = acc8; const double* yc = acc8 + 4;   // cubic coefficients, highest degree first
    // ---- curvature of the fitted cubics every 0.25 m, fitted by a cubic
    kc[0] = kc[1] = kc[2] = kc[3] = 0.0;
    for (int g = k; g < a.n2; g += 32) {
        const double tt = 0.25 * (double)g;
        const double dx = xc[2] + 2.0 * xc[1] * tt + 3.0 * xc[0] * (tt * tt), dy = yc[2] + 2.0 * yc[1] * tt + 3.0 * yc[0] * (tt * tt);
        const double ddx = 2.0 * xc[1] + 6.0 * xc[0] * tt, ddy = 2.0 * yc[1] + 6.0 * yc[0] * tt;
        const double Km = (dx * ddy - dy * ddx) / (dx * dx + dy * dy);
        for (int r = 0; r < 4; r++) kc[r] += a.P2[r * a.n2 + g] * Km;
    }
    S.template treduce<TeamSolver<1, 1>::OP_SUM, 2>(kc); S.template treduce<TeamSolver<1, 1>::OP_SUM, 2>(kc + 2);
    psi0 = atan2(yc[2], xc[2]);
    double sp0, cp0;
    mpc_sincos(psi0, &sp0, &cp0);
    ey = a.ey_from_path ? -(-sp0 * xw0 + cp0 * yw0) : 0.0;
}

MPC_DEV void rollout_group_frenet(const KCfg& cfg, const FrenetRolloutArgs& a, long b0, smem_t smem, smem_t px, int nwarps) {
    TeamSolver<1, 1> S(cfg, smem);
    const int k = S.k, N = cfg.N;
    const int w = thread_in_block() >> 5;
    const long b = b0 + w;
    const bool valid = b < a.B;
    const int pxw = SO(w * ROLLOUT_PX);
    const PathTable& path = a.paths[valid ? a.path_of[b] : 0];
    if (k < 8) sts(px, pxw + SO(k), (valid && k < 3) ? a.pose0[3 * b + k] : 0.0);
    double st[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    double acc_des = 0.0, df_des = 0.0, up_d = 0.0, up_a = 0.0;
    S.L.sx = S.L.sy = S.L.sp = S.L.sv = S.L.ua = S.L.ud = 0.0;   // start = 0.0, then the previous solution
    for (int t = 0; t < a.T; t++) {
        if (k == 0) { sts(px, pxw + SO(8), acc_des); sts(px, pxw + SO(9), df_des); }
        block_sync();
        if (thread_in_block() < nwarps) {   // lane = vehicle: ten 100 Hz publishes of ten Euler sub-steps each
            const int pv = SO(thread_in_block() * ROLLOUT_PX);
            double ps[8];
            for (int i = 0; i < 8; i++) ps[i] = lds(px, pv + SO(i));
            const double ad = lds(px, pv + SO(8)), dd = lds(px, pv + SO(9));
            MPC_NOUNROLL for (int i = 0; i < 10; i++) plant_step(ps, ad, dd);
            for (int i = 0; i < 8; i++) sts(px, pv + SO(i), ps[i]);
        }
        block_sync();
        if (!valid) continue;
        for (int i = 0; i < 8; i++) st[i] = lds(px, pxw + SO(i));
        // ---- the path ahead -> curvature polynomial, e_y, psi_start
        double kc[4], ey, psi0;
        frenet_reference(S, path, a, st[0], st[1], st[2], kc, ey, psi0);
        // ---- update_init_cond(0, e_y, -psi_start, v), update_reference(path, K_coeffs, des_speed), solve_model (:125-130)
        S.set_kpoly(kc[0], kc[1], kc[2], kc[3]);
        syncwarp();
        {
            const double cv[8] = {0.0, ey, -psi0, st[3], up_d, up_a, a.target_vel, 0.0};
            if (k < 8) sts(smem, SO(W_CONST + k), sel8(cv, k));
        }
        syncwarp();
        const Result r = S.solve();
        acc_des = shfl(S.L.ua, 0); df_des = shfl(S.L.ud, 0);   // published whatever the status (:139-143)
        up_d = df_des; up_a = acc_des;                           // update_current_input(df_opt, a_opt) (:145)
        if (a.log && k < 8) {
            const double lv[8] = {st[0], st[1], st[2], st[3], acc_des, df_des, (double)r.status, (double)r.iters};
            a.log[((long)t * a.B + b) * 8 + k] = sel8(lv, k);
        }
    }
    if (valid && a.final_state && k < 8) a.final_state[b * 8 + k] = sel8(st, k);
    block_sync();
}

}  // namespace mpcb200
