// mpcb_ocp.cuh - primal-dual interior-point solve of the dynamic OCP, stage-structured.
//
// Replaces `solver(lbx,ubx,x0,p,lbg,ubg)` at MPC_code.py:776-781 for the NLP that
// Control_Calc.py:20-260 builds (variables w=[x0,u0,...,xN], equality rows Fx(xk,uk)-x_{k+1},
// range rows Y_k in [ymin,ymax], box bounds), following IPOPT's algorithm (Waechter & Biegler
// 2006: monotone barrier, fraction-to-the-boundary, filter line search, delta_w inertia ladder).
// Instead of IPOPT's general sparse KKT factorisation the Newton system is solved by a Riccati
// recursion over the stages (x0 fixed and eliminated, range-row slacks and all bound multipliers
// condensed into the stage Hessians).
//
// Work split (one "tick" = the four kernels, each a thin wrapper around a function below):
//   ocp_eval_stage   one thread per (instance, stage): derivatives at the current iterate
//   ocp_kkt          per instance: optimality error, barrier update, Riccati solve, step sizes
//   ocp_trial_stage  one thread per (instance, stage): functions at the trial point
//   ocp_accept       per instance: filter test, accept (-> eval) or halve the step (-> trial)
// Every function is host/device so the identical code can be exercised on the CPU by the tests.
#pragma once
#include "mpcb_device.cuh"

#define NG   MPCB_NG
// The OCP may carry u_{k-1} as extra state components (Delta-u costs / Delta-u bounds, Control_Calc.py:163-169,
// 180-181): stage state z_k = [x_k; v_k], v_k = u_{k-1}, with the linear rows v_{k+1} = u_k.  NAUG = nu or 0.
#define NAUG MPCB_NAUG
#define NXA  (NX + NAUG)                  // stage state size seen by the Riccati recursion
#define NZA  (NXA + NU)
#define NZAP (NZA * (NZA + 1) / 2)
#define NXAP (NXA * (NXA + 1) / 2)
#define NWI  (NH * NZA + NXA)             // internal iterate [z_0,u_0,...,z_N]; the caller's w keeps the reference layout
#define NW   MPCB_NW
#define NPAR MPCB_NPAR
#define MPCB_MAXFILT 24

enum { ST_EVAL = 0, ST_LS = 1, ST_DONE = 2 };

struct IpmOpts {       // IPOPT option names; values set from mpcb_opts_t, the rest are IPOPT defaults
    int    max_iter;
    double tol, mu_init, bound_relax, bound_push, acceptable_tol;
    int    honor_original_bounds, acceptable_iter;
};

struct InstState {
    double mu, tau, alpha, alpha_z, theta, phi, gphid, amin, theta0, dw_last, fval, E0;
    double theta_entry;                   // violation at which the feasibility restoration was entered
    int    state, iter, status, nfilt, acc_cnt, ls_iter;
    int    resto, resto_calls;            // in restoration / number of times it was entered in this solve
    double filt[2 * MPCB_MAXFILT];
};

#if MPCB_CONTFORM
// ContForm (Control_Calc.py:102-111,153-158): the OCP integrates xdot = fx + px together with the quadrature of the
// stage cost; state [x; q], all other inputs frozen over the interval (time too - it is a parameter of the reference's
// integrator call).  DEVIATION: classic RK4 with MPCB_CMX sub-steps instead of SUNDIALS IDAS.
struct ContCtx { const double* u; const double* par; const double* pxk; const double* pyk; };
#ifndef MPCB_OCQ_NC
#define MPCB_OCQ_NC 0
#endif
#ifndef MPCB_OCQ_NR
#define MPCB_OCQ_NR 0
#endif
struct SysCont {
    static constexpr int NS = NX + 1, NM = MPCB_CMX, NC = MPCB_OCQ_NC, NR = MPCB_OCQ_NR;
    typedef ContCtx Ctx;
#if MPCB_OCQ_NC + MPCB_OCQ_NR > 0
    MPCB_HDM void f_c(const double* x, const Ctx& c, double, double* o, double* cache) { ocq_f_c(x, c.u, c.par, c.pxk, c.pyk, o, cache); }
    MPCB_HDM void f_rc(const double* x, const Ctx& c, double, const double* cache, double* o, double* rc) {
        ocq_f_rc(x, c.u, c.par, c.pxk, c.pyk, cache, o, rc);
    }
    MPCB_HDM void f_rcp(const double* x, const Ctx& c, double, const double* cache, double* rc) { ocq_f_rcp(x, c.u, c.par, c.pxk, c.pyk, cache, rc); }
    MPCB_HDM void f_vjp_c(const double* x, const Ctx& c, double, const double* nu, const double* cache, const double* rc, double* o) {
        ocq_f_vjp_c(x, c.u, c.par, c.pxk, c.pyk, nu, cache, rc, o);
    }
    MPCB_HDM void f_sh_c(const double* x, const Ctx& c, double, const double* S, const double* nu, const double* cache,
                         const double* rc, double* o, double* K, double* Hc) {
        ocq_f_sh_c(x, c.u, c.par, c.pxk, c.pyk, S, nu, cache, rc, o, K, Hc);
    }
#endif
    MPCB_HDM void f(const double* x, const Ctx& c, double, double* o) { ocq_f(x, c.u, c.par, c.pxk, c.pyk, o); }
    MPCB_HDM void f_vjp(const double* x, const Ctx& c, double, const double* nu, double* o) { ocq_f_vjp(x, c.u, c.par, c.pxk, c.pyk, nu, o); }
    MPCB_HDM void f_sh(const double* x, const Ctx& c, double, const double* S, const double* nu, double* o, double* K, double* Hc) {
        ocq_f_sh(x, c.u, c.par, c.pxk, c.pyk, S, nu, o, K, Hc);
    }
};
#endif

// Per-instance view of the solver workspace (all device pointers).
struct OcpInst {
    double* w; double* wext; const double* par;      // w: internal iterate (NWI); wext: caller buffer (NW, reference layout)
    double *lam, *lamn, *s, *ds, *ym, *dym, *zL, *zU, *vL, *vU, *dw;
    double *rec, *trec, *frec, *partt, *nuT, *nuTn;
    InstState* st;
};
struct OcpShared { const double *lbx, *ubx, *lbg, *ubg; IpmOpts o; };

// ---- per-stage records ------------------------------------------------------------------------
// k_ocp_eval condenses everything the Newton step needs from stage k into ONE contiguous record, so that the
// sequential sweeps of the KKT step stream memory instead of gathering from a dozen arrays:
#define NGS (NG > 0 ? NG : 1)
#define R_AB   0                          // NXA*NZA  [A_k | B_k], column-major
#define R_C    (R_AB + NXA * NZA)           // NXA     defect  Fx(x_k,u_k) - x_{k+1}
#define R_M    (R_C + NXA)                 // NZA*NZA  H_k + diag(zL/dL + zU/dU) + G' Sigma_s G   (delta_w = 0)
#define R_GL   (R_M + NZA * NZA)            // NZA     gradient of the stage cost
#define R_IL   (R_GL + NZA)                // NZA     1 / (v - lo)  (0: no lower bound / fixed x_0)
#define R_IU   (R_IL + NZA)                // NZA     1 / (hi - v)
#define R_G    (R_IU + NZA)                // NG*NZA  Jacobian of the range rows (column-major NG x NZA)
#define R_SG   (R_G + NGS * NZA)           // NG     Sigma_s = vL/(s-lo) + vU/(hi-s)
#define R_ISL  (R_SG + NGS)               // NG     1 / (s - lo)
#define R_ISU  (R_ISL + NGS)              // NG     1 / (hi - s)
#define R_RG   (R_ISU + NGS)              // NG     g - s
#define R_BWD  (R_RG + NGS)               // ---- everything above is what the backward sweep stages (one burst);
                                          //      the stage-parallel pass reads R_GL .. R_GV (one burst); order matters
#define R_QL   R_BWD                      // NZA     (1/(v-lo)) / zL   (0: no bound) - keeps the step-size rules division free
#define R_QU   (R_QL + NZA)                // NZA     (1/(hi-v)) / zU
#define R_QSL  (R_QU + NZA)                // NG     (1/(s-lo)) / vL
#define R_QSU  (R_QSL + NGS)              // NG     (1/(hi-s)) / vU
#define R_YM   (R_QSU + NGS)              // NG     multiplier of the range row
#define R_GV   (R_YM + NGS)               // NG     g
#define R_PART (R_GV + NGS)               // 10: cost, theta, dual_max, prim_max, ysum, zsum, nb, pmin, pmax, sum log(slack)
#define NPART  10
#define REC_SZ ((R_PART + NPART + 1) / 2 * 2)
// terminal equality E x_N = x_s (TermCons, Control_Calc.py:197-198): NXT rows, multiplier nuT
#ifndef MPCB_TERMCONS
#define MPCB_TERMCONS 0
#endif
#define NXT (MPCB_TERMCONS ? NX : 0)
// terminal record (x_N)
#define T_H    0                          // NXA*NXA  Hessian of the terminal cost
#define T_GN   (NXA * NXA)                  // NXA     its gradient
#define T_IL   (T_GN + NXA)
#define T_IU   (T_IL + NXA)
#define T_ZL   (T_IU + NXA)
#define T_ZU   (T_ZL + NXA)
#define T_QL   (T_ZU + NXA)
#define T_QU   (T_QL + NXA)
#define T_RT   (T_QU + NXA)                 // NXT     residual of the terminal equality
#define T_PART (T_RT + NXT)                // 10: V, theta_T, dual_max, prim_T, |nuT|_1, zsum, nb, pmin, pmax, sum log(slack)
#define TREC_SZ ((T_PART + NPART + 1) / 2 * 2)
// forward records written by the Riccati sweep
#define FREC_K   0
#define FREC_KF  (NU * NXA)
#define FREC_GA  (FREC_KF + NU)            // NU*NXT   Gamma_k: du_k += Gamma_k nuT   (terminal equality)
#define FREC_P   (FREC_GA + NU * NXT)
#define FREC_PV  (FREC_P + NXA * NXA)
#define FREC_PI  (FREC_PV + NXA)           // NXA*NXT  Pi_{k+1}: lam_k += Pi_{k+1} nuT
#define FREC_SZ  ((FREC_PI + NXA * NXT + 1) / 2 * 2)

struct OcpLayout {
    static constexpr int lam = 0;
    static constexpr int lamn = lam + NH * NXA;
    static constexpr int s = lamn + NH * NXA;
    static constexpr int ds = s + NH * NGS;
    static constexpr int ym = ds + NH * NGS;
    static constexpr int dym = ym + NH * NGS;
    static constexpr int vL = dym + NH * NGS;
    static constexpr int vU = vL + NH * NGS;
    static constexpr int zL = vU + NH * NGS;
    static constexpr int zU = zL + NWI;
    static constexpr int dw = zU + NWI;
    static constexpr int wint = (dw + NWI + 1) / 2 * 2;
    static constexpr int rec = (wint + NWI + 1) / 2 * 2;
    static constexpr int trec = rec + NH * REC_SZ;
    static constexpr int frec = trec + TREC_SZ;
    static constexpr int partt = frec + NH * FREC_SZ;
    static constexpr int nuT = (partt + (NH + 1) * 4 + 1) / 2 * 2;      // multiplier of the terminal equality and its new value
    static constexpr int nuTn = nuT + NXT;
    static constexpr int total = (nuTn + NXT + 1) / 2 * 2;
};

MPCB_HD OcpInst ocp_inst(double* ws, double* wext, const double* par, InstState* st) {
    OcpInst I;
    I.w = ws + OcpLayout::wint; I.wext = wext; I.par = par; I.st = st;
    I.lam = ws + OcpLayout::lam; I.lamn = ws + OcpLayout::lamn; I.s = ws + OcpLayout::s; I.ds = ws + OcpLayout::ds;
    I.ym = ws + OcpLayout::ym; I.dym = ws + OcpLayout::dym; I.vL = ws + OcpLayout::vL; I.vU = ws + OcpLayout::vU;
    I.zL = ws + OcpLayout::zL; I.zU = ws + OcpLayout::zU; I.dw = ws + OcpLayout::dw;
    I.rec = ws + OcpLayout::rec; I.trec = ws + OcpLayout::trec; I.frec = ws + OcpLayout::frec;
    I.partt = ws + OcpLayout::partt; I.nuT = ws + OcpLayout::nuT; I.nuTn = ws + OcpLayout::nuTn;
    return I;
}

// ---- bounds ---------------------------------------------------------------------------------
MPCB_HD bool fin(double v) { return v > -1e300 && v < 1e300; }
MPCB_HD double rlo(double lo, double f) { return lo - f * fmax(1.0, fabs(lo)); }
MPCB_HD double rhi(double hi, double f) { return hi + f * fmax(1.0, fabs(hi)); }

// IPOPT's initial push of a primal value into its (relaxed) bounds: bound_push / bound_frac.
MPCB_HD double push_in(double v, double lo, double hi, double kappa) {
    const bool hl = fin(lo), hu = fin(hi);
    if (hl) {
        double pl = kappa * fmax(1.0, fabs(lo));
        if (hu) pl = fmin(pl, kappa * (hi - lo));
        v = fmax(v, lo + pl);
    }
    if (hu) {
        double pu = kappa * fmax(1.0, fabs(hi));
        if (hl) pu = fmin(pu, kappa * (hi - lo));
        v = fmin(v, hi - pu);
    }
    return v;
}

MPCB_HD void stage_params(const double* par, int k, double* d, double* px, double* py, double* t0) {
MPCB_UNROLL
    for (int i = 0; i < ND; ++i) d[i] = par[MPCB_OFF_D + i];
MPCB_UNROLL
    for (int i = 0; i < NPX; ++i) px[i] = par[MPCB_OFF_PX + k * NPX + i];
MPCB_UNROLL
    for (int i = 0; i < NPY; ++i) py[i] = par[MPCB_OFF_PY + k * NPY + i];
    *t0 = par[MPCB_OFF_T];
}

// =============================================================================================
// init: starting point (IPOPT default initialisation), one call per (instance, stage k=0..NH).
// Copies the caller's guess (reference layout) into the internal iterate z_k = [x_k; v_k], u_k.
// =============================================================================================
MPCB_HD double init_push(const OcpShared& S, int wi, double v) {       // push component wi of the internal iterate inside
    const double rf = S.o.bound_relax, lo = S.lbx[wi], hi = S.ubx[wi];
    return push_in(v, fin(lo) ? rlo(lo, rf) : lo, fin(hi) ? rhi(hi, rf) : hi, S.o.bound_push);
}

MPCB_HD void ocp_init_stage(OcpInst& I, const OcpShared& S, int k) {
    const double rf = S.o.bound_relax, kp = S.o.bound_push;
    double* w = I.w;
    const double* we = I.wext;
    if (k == 0) {
        InstState& st = *I.st;
        st.mu = S.o.mu_init; st.tau = fmax(0.99, 1.0 - S.o.mu_init);
        st.alpha = st.alpha_z = 0.0; st.theta0 = -1.0; st.dw_last = 0.0; st.fval = 0.0; st.E0 = 0.0;
        st.state = ST_EVAL; st.iter = 0; st.status = -1; st.nfilt = 0; st.acc_cnt = 0; st.ls_iter = 0;
        st.resto = 0; st.resto_calls = 0; st.theta_entry = 0.0;
        // a non-finite estimate / target / disturbance (diverged instance) cannot be evaluated: IPOPT's
        // Invalid_Number_Detected (-13), decided here so that the instance does not burn line-search ticks
        double chk = 0.0;
        for (int i = 0; i < MPCB_OFF_LAM; ++i) chk += I.par[i];
        if (!(chk == chk) || !fin(chk)) { st.state = ST_DONE; st.status = -13; }
        for (int i = 0; i < NXT; ++i) I.nuT[i] = 0.0;
    }
    // state part z_k = [x_k; v_k]
    for (int i = 0; i < NXA; ++i) {
        const int wi = k * NZA + i;
        double v;
        if (i < NX) v = (k == 0) ? I.par[MPCB_OFF_X0 + i] : we[k * NZ + i];                     // MPC_code.py:734
        else v = (k == 0) ? I.par[MPCB_OFF_UM1 + (i - NX)]                                      // Control_Calc.py:163-164
                          : init_push(S, (k - 1) * NZA + NXA + (i - NX), we[(k - 1) * NZ + NX + (i - NX)]);   // = pushed u_{k-1}
        if (k == 0) { w[wi] = v; I.zL[wi] = 0.0; I.zU[wi] = 0.0; continue; }                    // z_0 is fixed
        w[wi] = init_push(S, wi, v);
        I.zL[wi] = fin(S.lbx[wi]) ? 1.0 : 0.0;
        I.zU[wi] = fin(S.ubx[wi]) ? 1.0 : 0.0;
    }
    if (k < NH) {
        for (int i = 0; i < NU; ++i) {
            const int wi = k * NZA + NXA + i;
            w[wi] = init_push(S, wi, we[k * NZ + NX + i]);
            I.zL[wi] = fin(S.lbx[wi]) ? 1.0 : 0.0;
            I.zU[wi] = fin(S.ubx[wi]) ? 1.0 : 0.0;
        }
MPCB_UNROLL
        for (int i = 0; i < NXA; ++i) I.lam[k * NXA + i] = 0.0;
#if NG > 0
        double d[ND + 1], px[NPX + 1], py[NPY + 1], t0, Y[NG];
        stage_params(I.par, k, d, px, py, &t0);
        ocp_out(w + k * NZA, w + k * NZA + NXA, I.par, px, py, Y);
        for (int i = 0; i < NG; ++i) {
            const double lo = S.lbg[k * NG + i], hi = S.ubg[k * NG + i];
            const double lor = fin(lo) ? rlo(lo, rf) : lo, hir = fin(hi) ? rhi(hi, rf) : hi;
            I.s[k * NG + i] = push_in(Y[i], lor, hir, kp);
            I.ym[k * NG + i] = 0.0;
            I.vL[k * NG + i] = fin(lo) ? 1.0 : 0.0;
            I.vU[k * NG + i] = fin(hi) ? 1.0 : 0.0;
        }
#endif
    }
}

// copy the internal iterate back into the caller's buffer (reference layout)
MPCB_HD void ocp_export_stage(OcpInst& I, int k) {
    for (int i = 0; i < NX; ++i) I.wext[k * NZ + i] = I.w[k * NZA + i];
    if (k < NH) for (int i = 0; i < NU; ++i) I.wext[k * NZ + NX + i] = I.w[k * NZA + NXA + i];
}

// =============================================================================================
// eval: derivatives of stage k at the current iterate, condensed into the stage record
// (k = 0..NH-1; k = NH-1 also writes the terminal record)
// =============================================================================================
// rmu > 0: restoration mode - the multipliers are not iterated, the primal barrier Hessian mu / d^2 is used (z = mu / d)
MPCB_HD void bound_terms(double v, double lo, double hi, double zl, double zu, double rf, bool active, double rmu,
                         double* iL, double* iU, double* zL, double* zU, double* qL, double* qU, double* sig,
                         double* zsum, double* nb, double* pmin, double* pmax, double* prod) {
    *iL = *iU = *zL = *zU = *qL = *qU = 0.0;
    if (!active) return;
    if (fin(lo)) { const double d = v - rlo(lo, rf); const double id = MPCB_RCP(d); if (rmu > 0.0) zl = rmu * id;
                   *iL = id; *zL = zl; *qL = id * MPCB_RCP(zl); *sig += zl * id;
                   *zsum += zl; *nb += 1.0; *pmin = fmin(*pmin, d * zl); *pmax = fmax(*pmax, d * zl); *prod *= d; }
    if (fin(hi)) { const double d = rhi(hi, rf) - v; const double id = MPCB_RCP(d); if (rmu > 0.0) zu = rmu * id;
                   *iU = id; *zU = zu; *qU = id * MPCB_RCP(zu); *sig += zu * id;
                   *zsum += zu; *nb += 1.0; *pmin = fmin(*pmin, d * zu); *pmax = fmax(*pmax, d * zu); *prod *= d; }
}

// sub-step records of the RK4 sweeps: the model's, or the cost-augmented system's for ContForm problems
#if MPCB_CONTFORM
#define EVAL_RK_DOUBLES (RkSize<SysCont>::TOTAL)
#elif MPCB_DYN_RK4
#define EVAL_RK_DOUBLES (RkSize<SysModel>::TOTAL)
#else
#define EVAL_RK_DOUBLES 0
#endif

// FIRST: the evaluation that follows ocp_init_stage.  Every multiplier is zero there, so the Hessian of the Lagrangian is
// the cost Hessian alone and the adjoint / second-order RK4 sweeps would only add exact zeros: the dynamics are
// differentiated to first order (dyn_sens, one forward sweep, no sub-step records).  RK4 models with a separate stage
// cost only (the quadrature form integrates the cost with the adjoint seed 1).
#ifndef MPCB_EVAL_FIRST
#define MPCB_EVAL_FIRST (MPCB_DYN_RK4 && !MPCB_CONTFORM && !MPCB_DENSE_SH)
#endif
template <bool EXT = false, bool FIRST = false>
MPCB_HD void ocp_eval_stage(OcpInst& I, const OcpShared& S, int k, RkBuf rb = RkBuf{nullptr, 1}) {
    const double* w = I.w;
    const double rf = S.o.bound_relax;
    double z[NXA], u[NU], lam[NXA], d[ND + 1], px[NPX + 1], py[NPY + 1], t0;
MPCB_UNROLL
    for (int i = 0; i < NXA; ++i) { z[i] = w[k * NZA + i]; lam[i] = I.lam[k * NXA + i]; }
MPCB_UNROLL
    for (int i = 0; i < NU; ++i) u[i] = w[k * NZA + NXA + i];
    stage_params(I.par, k, d, px, py, &t0);
    double xn[NXA], A[NXA * NXA], Bm[NXA * NU], Hp[NZAP], l, g[NZA];
    ocp_cost_d(z, u, I.par, px, py, &l, g, Hp);          // Hp <- cost Hessian, then accumulate the rest
#if MPCB_CONTFORM
    {   // dynamics and stage cost from one sweep over [x; q] with the adjoint seed [lam; 1]
        constexpr int NS = NX + 1, NZS = NS + NU;
        ContCtx cc; cc.u = u; cc.par = I.par; cc.pxk = px; cc.pyk = py;
        double xt[NS], lt[NS], xe[NS], S[NS * NZS], Ht[NZS * (NZS + 1) / 2];
MPCB_UNROLL
        for (int i = 0; i < NX; ++i) { xt[i] = z[i]; lt[i] = lam[i]; }
        xt[NX] = 0.0; lt[NX] = 1.0;
MPCB_UNROLL
        for (int i = 0; i < NZS * (NZS + 1) / 2; ++i) Ht[i] = 0.0;
        if constexpr (EXT) {
            rk4_full_t<SysCont>(xt, cc, t0, lt, xe, S, Ht, rb);
        } else {
            double lbuf[RkSize<SysCont>::TOTAL];
            rk4_full_t<SysCont>(xt, cc, t0, lt, xe, S, Ht, RkBuf{lbuf, 1});
        }
        l = xe[NX];
MPCB_UNROLL
        for (int j = 0; j < NZ; ++j) {
            const int js = (j < NX) ? j : j + 1;          // skip the q0 column
            g[j] = S[NX + NS * js];
MPCB_UNROLL
            for (int i = 0; i < NX; ++i) { if (j < NX) A[i + NX * j] = S[i + NS * js]; else Bm[i + NX * (j - NX)] = S[i + NS * js]; }
MPCB_UNROLL
            for (int i = 0; i <= j; ++i) { const int is = (i < NX) ? i : i + 1; Hp[tri(j, i)] += Ht[tri(js, is)]; }
        }
MPCB_UNROLL
        for (int i = 0; i < NX; ++i) xn[i] = xe[i];
    }
#elif NAUG == 0
    if constexpr (FIRST) dyn_sens(z, u, d, px, t0, xn, A, Bm);
    else dyn_full<EXT>(z, u, d, px, t0, lam, xn, A, Bm, Hp, rb);
#else
    {   // model part by the RK4 sweeps, then embedded into the augmented stage:  z+ = [Fx(x,u); u]
        double xm[NX], Am[NX * NX], Bmm[NX * NU], Hm[NZP];
MPCB_UNROLL
        for (int i = 0; i < NZP; ++i) Hm[i] = 0.0;
        if constexpr (FIRST) dyn_sens(z, u, d, px, t0, xm, Am, Bmm);
        else dyn_full<EXT>(z, u, d, px, t0, lam, xm, Am, Bmm, Hm, rb);
MPCB_UNROLL
        for (int i = 0; i < NXA * NXA; ++i) A[i] = 0.0;
MPCB_UNROLL
        for (int i = 0; i < NXA * NU; ++i) Bm[i] = 0.0;
MPCB_UNROLL
        for (int j = 0; j < NX; ++j)
MPCB_UNROLL
            for (int i = 0; i < NX; ++i) A[i + NXA * j] = Am[i + NX * j];
MPCB_UNROLL
        for (int j = 0; j < NU; ++j) {
MPCB_UNROLL
            for (int i = 0; i < NX; ++i) Bm[i + NXA * j] = Bmm[i + NX * j];
            Bm[NX + j + NXA * j] = 1.0;
        }
MPCB_UNROLL
        for (int i = 0; i < NX; ++i) xn[i] = xm[i];
MPCB_UNROLL
        for (int i = 0; i < NU; ++i) xn[NX + i] = u[i];
        // model Hessian (ordering x,u) into the augmented ordering (x, v, u)
MPCB_UNROLL
        for (int i = 0; i < NZ; ++i)
MPCB_UNROLL
            for (int j = 0; j <= i; ++j) {
                const int ia = (i < NX) ? i : i + NAUG, ja = (j < NX) ? j : j + NAUG;
                Hp[tri(ia, ja)] += Hm[tri(i, j)];
            }
    }
#endif
#ifndef MPCB_VEC_REC
#define MPCB_VEC_REC 1
#endif
#if MPCB_VEC_REC
    double r[REC_SZ];          // the record is assembled in registers and written out with 128-bit stores at the end
#else
    double* r = I.rec + k * REC_SZ;
#endif
    // Feasibility restoration (entered by ocp_accept when the line search fails): the step minimises
    //   zeta/2 |D_R dv|^2 - mu sum log(slacks to the bounds)   subject to the linearised constraints,
    // zeta = sqrt(mu), D_R = diag(1 / max(1, |v|)): no cost gradient, Hessian zeta D_R^2, primal barrier terms.
    const bool resto = I.st->resto != 0;
    const double rmu = resto ? I.st->mu : 0.0, zeta = resto ? sqrt(I.st->mu) : 0.0;
    if (resto) {
MPCB_UNROLL
        for (int i = 0; i < NZAP; ++i) Hp[i] = 0.0;
MPCB_UNROLL
        for (int j = 0; j < NZA; ++j) {
            const double vj = w[k * NZA + j], sc = fmax(1.0, fabs(vj));
            Hp[tri(j, j)] = zeta / (sc * sc);
            g[j] = 0.0;
        }
    }
    double th = 0.0, prim = 0.0, ysum = 0.0, zsum = 0.0, nb = 0.0, pmin = 1e300, pmax = -1e300;
    double prod = 1.0;     // product of all slacks-to-bounds of the stage: one log instead of one per bound
MPCB_UNROLL
    for (int i = 0; i < NXA; ++i) {
        const double ci = xn[i] - w[(k + 1) * NZA + i];
        r[R_C + i] = ci;
        th += fabs(ci); prim = fmax(prim, fabs(ci)); ysum += fabs(lam[i]);
    }
    // dual residual of the stage variables, started with the cost gradient and the dynamics multipliers
    double res[NZA], dg[NZA];
MPCB_UNROLL
    for (int j = 0; j < NZA; ++j) {
        double a = g[j];
MPCB_UNROLL
        for (int i = 0; i < NXA; ++i) a += ((j < NXA) ? A[i + NXA * j] : Bm[i + NXA * (j - NXA)]) * lam[i];
        if (j < NXA && k > 0) a -= I.lam[(k - 1) * NXA + j];
        res[j] = a; dg[j] = 0.0;
    }
MPCB_UNROLL
    for (int j = 0; j < NZA; ++j) {
        const int wi = k * NZA + j;
        const bool active = !(k == 0 && j < NXA);          // x_0 is fixed
        double iL, iU, zL, zU, qL, qU;
        bound_terms(w[wi], S.lbx[wi], S.ubx[wi], I.zL[wi], I.zU[wi], rf, active, rmu, &iL, &iU, &zL, &zU, &qL, &qU, &dg[j], &zsum, &nb, &pmin, &pmax, &prod);
        r[R_IL + j] = iL; r[R_IU + j] = iU; r[R_QL + j] = qL; r[R_QU + j] = qU; r[R_GL + j] = g[j];
        res[j] += zU - zL;
    }
    double M[NZA * NZA], dual_s = 0.0;
MPCB_UNROLL
    for (int j = 0; j < NZA; ++j)
MPCB_UNROLL
        for (int i = 0; i < NZA; ++i) M[i + NZA * j] = Hp[tri(i, j)] + (i == j ? dg[j] : 0.0);
#if NG > 0
    {
        double Y[NG], JY[NG * NZA], HY[NZAP], mult[NG];
MPCB_UNROLL
        for (int i = 0; i < NG; ++i) mult[i] = I.ym[k * NG + i];
        ocp_out_d(z, u, I.par, px, py, mult, Y, JY, HY);
#if !MPCB_OUT_LINEAR
        if (!resto) {
MPCB_UNROLL
            for (int j = 0; j < NZA; ++j)
MPCB_UNROLL
                for (int i = 0; i < NZA; ++i) M[i + NZA * j] += HY[tri(i, j)];
        }
#endif
MPCB_UNROLL
        for (int q = 0; q < NG; ++q) {
            const int gi = k * NG + q;
            const double sv = I.s[gi], lo = S.lbg[gi], hi = S.ubg[gi];
            double isl, isu, vl, vu, qsl, qsu, sig = 0.0;
            bound_terms(sv, lo, hi, I.vL[gi], I.vU[gi], rf, true, rmu, &isl, &isu, &vl, &vu, &qsl, &qsu, &sig, &zsum, &nb, &pmin, &pmax, &prod);
            if (resto) { const double sc = fmax(1.0, fabs(sv)); sig += zeta / (sc * sc); }
            const double rg = Y[q] - sv;
            r[R_SG + q] = sig; r[R_ISL + q] = isl; r[R_ISU + q] = isu;
            r[R_QSL + q] = qsl; r[R_QSU + q] = qsu;
            r[R_RG + q] = rg; r[R_YM + q] = mult[q]; r[R_GV + q] = Y[q];
            th += fabs(rg); prim = fmax(prim, fabs(rg)); ysum += fabs(mult[q]);
            dual_s = fmax(dual_s, fabs(-mult[q] - vl + vu));   // dual residual of the slack
MPCB_UNROLL
            for (int j = 0; j < NZA; ++j) {
                r[R_G + q + NG * j] = JY[q + NG * j];
                res[j] += JY[q + NG * j] * mult[q];
MPCB_UNROLL
                for (int i = 0; i < NZA; ++i) M[i + NZA * j] += JY[q + NG * i] * sig * JY[q + NG * j];
            }
        }
    }
#endif
    double dual = dual_s;
MPCB_UNROLL
    for (int j = 0; j < NZA; ++j) if (!(k == 0 && j < NXA)) dual = fmax(dual, fabs(res[j]));
MPCB_UNROLL
    for (int i = 0; i < NXA * NXA; ++i) r[R_AB + i] = A[i];
MPCB_UNROLL
    for (int i = 0; i < NXA * NU; ++i) r[R_AB + NXA * NXA + i] = Bm[i];
MPCB_UNROLL
    for (int i = 0; i < NZA * NZA; ++i) r[R_M + i] = M[i];
    r[R_PART + 0] = l; r[R_PART + 1] = th; r[R_PART + 2] = dual; r[R_PART + 3] = prim; r[R_PART + 4] = ysum;
    r[R_PART + 5] = zsum; r[R_PART + 6] = nb; r[R_PART + 7] = pmin; r[R_PART + 8] = pmax; r[R_PART + 9] = log(prod);
#if MPCB_VEC_REC
    {
        double* rg_ = I.rec + k * REC_SZ;               // 16-byte aligned: REC_SZ and the workspace offsets are even
#ifdef __CUDA_ARCH__
MPCB_UNROLL
        for (int i = 0; i < (R_PART + NPART + 1) / 2; ++i)
            reinterpret_cast<double2*>(rg_)[i] = make_double2(r[2 * i], (2 * i + 1 < R_PART + NPART) ? r[2 * i + 1] : 0.0);
#else
        for (int i = 0; i < R_PART + NPART; ++i) rg_[i] = r[i];
#endif
    }
#endif
    if (k == NH - 1) {
        double V, gN[NX], HN[NXP_ + 1];
        double* t = I.trec;
        ocp_term_d(w + NH * NZA, I.par, &V, gN, HN);           // terminal cost acts on x_N only (Control_Calc.py:194-196,209)
        double dualN = 0.0, zs = 0.0, nbn = 0.0, pmn = 1e300, pmx = -1e300, prodN = 1.0;
MPCB_UNROLL
        for (int j = 0; j < NXA; ++j) {
            const int wi = NH * NZA + j;
            double iL, iU, zL, zU, qL, qU, sig = 0.0;
            bound_terms(w[wi], S.lbx[wi], S.ubx[wi], I.zL[wi], I.zU[wi], rf, true, rmu, &iL, &iU, &zL, &zU, &qL, &qU, &sig, &zs, &nbn, &pmn, &pmx, &prodN);
            const double gj = (resto || j >= NX) ? 0.0 : gN[j];
            t[T_IL + j] = iL; t[T_IU + j] = iU; t[T_ZL + j] = zL; t[T_ZU + j] = zU; t[T_QL + j] = qL; t[T_QU + j] = qU; t[T_GN + j] = gj;
            double dr = gj - lam[j] + zU - zL;                           // lam = lam_N for k = NH-1
#if MPCB_TERMCONS
            if (j < NX) dr += I.nuT[j];
#endif
            dualN = fmax(dualN, fabs(dr));
MPCB_UNROLL
            for (int i = 0; i < NXA; ++i) {
                double hij = (i < NX && j < NX) ? HN[tri(i, j)] : 0.0;
                if (resto) { const double sc = fmax(1.0, fabs(w[wi])); hij = (i == j) ? zeta / (sc * sc) : 0.0; }
                t[T_H + i + NXA * j] = hij;
            }
        }
        double thT = 0.0, primT = 0.0, ysT = 0.0;
#if MPCB_TERMCONS
        {
            double rT[NX];
            ocp_termc(w + NH * NZA, I.par, rT);
            for (int j = 0; j < NX; ++j) { t[T_RT + j] = rT[j]; thT += fabs(rT[j]); primT = fmax(primT, fabs(rT[j])); ysT += fabs(I.nuT[j]); }
        }
#endif
        t[T_PART + 0] = V; t[T_PART + 1] = thT; t[T_PART + 2] = dualN; t[T_PART + 3] = primT; t[T_PART + 4] = ysT;
        t[T_PART + 5] = zs; t[T_PART + 6] = nbn; t[T_PART + 7] = pmn; t[T_PART + 8] = pmx; t[T_PART + 9] = log(prodN);
    }
}

// =============================================================================================
// Lane-generic helpers.  ocp_kkt / ocp_accept are written once over a lane group (Lanes<L>, mpcb_device.cuh) and run
// either by MPCB_KKT_LANES = 32 lanes of a warp (lanes strided over matrix entries, reductions by shuffle, per-warp
// scratch in shared memory: the mapping for large stage blocks), by one device thread per instance (MPCB_KKT_LANES = 1:
// everything in registers, records read in place - the mapping for small systems such as Ex_NMPC), or by a single host
// "lane" (tests).
// =============================================================================================
// Measured on B200 at 4 096 instances (profiles/r01_variants.txt): one warp per instance is faster than one thread per
// instance (the latter has 5x fewer instructions but only 128 warps to hide latency with); the thread mapping is the
// one to pick for very large batches and is kept selectable at build time (-DMPCB_KKT_LANES=1).
#ifndef MPCB_KKT_LANES
#  define MPCB_KKT_LANES 32
#endif
// MPCB_KKT_LANES is one of 1, 2, 4, 8, 16, 32: with L < 32 a warp carries 32/L instances ("lane groups"); the stage
// blocks of small systems (Ex_NMPC: 3 x 5) leave most of 32 lanes idle, and the kernel is bound by issue slots.  The
// 32/L scratches of a warp share the 48 kB of static shared memory, so lane groups only build for problems whose
// KktScratch is small enough (mpcb_api.cu refuses the others: syn_12_4_20 at 4 lanes, syn_20_6_20 at 16 lanes or fewer
// - the latter builds with 32 lanes or with one thread per instance, whose scratch is thread-local).
#if MPCB_KKT_LANES != 1 && MPCB_KKT_LANES != 2 && MPCB_KKT_LANES != 4 && MPCB_KKT_LANES != 8 && \
    MPCB_KKT_LANES != 16 && MPCB_KKT_LANES != 32
#  error "MPCB_KKT_LANES must be one of 1, 2, 4, 8, 16, 32 (the lane-group masks and reductions assume a power of two <= 32)"
#endif
typedef Lanes<MPCB_KKT_LANES> KktLanes;       // ocp_riccati, ocp_kkt, ocp_sens_factor
typedef Lanes<32> WarpLanes;                  // ocp_accept: one whole warp per instance
#define KKT_STAGED (MPCB_KKT_LANES > 1)        // records staged through the scratch (lane mappings) or read in place

// scratch (doubles): shared memory per warp with 32 lanes, thread-local (registers) with one lane
// Record streaming of the lane mappings on the device: bulk asynchronous copies (cp.async.bulk, the TMA engine; SASS
// UBLKCP) from the workspace straight into a ring of KKT_NBUF shared-memory buffers, completion signalled on one mbarrier
// per buffer, issued KKT_NBUF - 1 stages ahead of the stage being processed.  Round 1 staged the next record through
// registers (one stage ahead): a third of the kernel's stall samples sat on that copy (profiles/r02_v2_sass_k_ocp_kkt.txt).
#define KKT_RBUF ((R_BWD + 1) / 2 * 2)          // doubles per ring buffer: a 16-byte multiple
#define KKT_NBUF (KKT_RBUF > 600 ? 2 : 3)       // large stage blocks: two buffers (the scratch must fit 48 kB of static shared memory)
struct KktScratch {
    static constexpr int R = 0;                                     // staged records (lane mappings only): KKT_NBUF buffers
    static constexpr int BAR = R + (KKT_STAGED ? KKT_NBUF * KKT_RBUF : 0);   // KKT_NBUF mbarriers (8 bytes each)
    static constexpr int P = BAR + (KKT_STAGED ? (KKT_NBUF + 1) / 2 * 2 : 0);   // NXA x NXA  cost-to-go Hessian of the next stage
    static constexpr int p = P + NXA * NXA;             // NXA
    static constexpr int M = p + NXA;                  // NZA x NZA  condensed stage Hessian
    static constexpr int q = M + NZA * NZA;             // NZA
    static constexpr int T = q + NZA;                  // NXA x NZA  P [A B]
    static constexpr int f = T + NXA * NZA;             // NXA       P c + p
    static constexpr int K = f + NXA;                  // NU x NXA
    static constexpr int kk = K + NU * NXA;            // NU
    static constexpr int cf = kk + NU;                // NGS      slack gradient coefficient
    static constexpr int F = cf + NGS;                // staged forward record (32-lane mapping only)
    static constexpr int dx = F + (KKT_STAGED ? FREC_SZ : 0);   // NXA
    static constexpr int du = dx + NXA;                // NU
    static constexpr int dxn = du + NU;               // NXA
    // terminal equality: Pi (two buffers), B'Pi, Gamma, Gramian G, free response h, multiplier nu
    static constexpr int PiA = dxn + NXA;             // NXA x NXT
    static constexpr int PiB = PiA + NXA * NXT;
    static constexpr int BtPi = PiB + NXA * NXT;      // NU x NXT
    static constexpr int Ga = BtPi + NU * NXT;        // NU x NXT
    static constexpr int Gm = Ga + NU * NXT;          // NXT x NXT
    static constexpr int hT = Gm + NXT * NXT;         // NXT
    static constexpr int nuS = hT + NXT;              // NXT
    static constexpr int total = (nuS + NXT + 1) / 2 * 2;           // even: every instance's scratch stays 16-byte aligned
};

#if defined(__CUDA_ARCH__) && KKT_STAGED
#define KKT_USE_TMA 1
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(void* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, void* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(void* bar, unsigned parity) {
    asm volatile("{\n .reg .pred p;\n WAIT_LOOP:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra WAIT_DONE;\n"
                 " bra WAIT_LOOP;\n WAIT_DONE:\n }" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// Ring of record buffers of one instance (one lane group).  `phase` holds the parity of every buffer's next completion.
struct RecRing {
    double* buf; unsigned long long* bar; unsigned phase;
    __device__ __forceinline__ void init(double* sm, int lane) {
        buf = sm + KktScratch::R; bar = reinterpret_cast<unsigned long long*>(sm + KktScratch::BAR); phase = 0u;
        if (lane == 0) {
            for (int b = 0; b < KKT_NBUF; ++b) mbar_init(bar + b, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    }
    // queue the copy of n0 doubles from g0 (and n1 from g1, placed after the first n0) into buffer b; one lane calls it
    __device__ __forceinline__ void issue(int b, const double* g0, int n0, const double* g1, int n1) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // earlier reads of this buffer precede the overwrite
        mbar_expect_tx(bar + b, 8u * (unsigned)(n0 + n1));
        bulk_g2s(buf + b * KKT_RBUF, g0, 8u * (unsigned)n0, bar + b);
        if (n1 > 0) bulk_g2s(buf + b * KKT_RBUF + n0, g1, 8u * (unsigned)n1, bar + b);
    }
    // every lane: wait for buffer b
    __device__ __forceinline__ const double* wait(int b) {
        mbar_wait(bar + b, (phase >> b) & 1u);
        phase ^= 1u << b;
        return buf + b * KKT_RBUF;
    }
};
#else
#define KKT_USE_TMA 0
#endif

#if KKT_USE_TMA
typedef RecRing KktIo;
#else
struct KktIo { int unused; };
#endif

// Riccati backward sweep with regularisation dw on every primal variable (and slack).  Returns false when
// some R_k + B_k' P_{k+1} B_k is not positive definite (wrong inertia).
MPCB_HD bool ocp_riccati(OcpInst& I, double mu, double dwreg, double* sm, KktIo& io) {
    const int lane = KktLanes::id();
    double* P = sm + KktScratch::P; double* p = sm + KktScratch::p; double* M = sm + KktScratch::M;
    double* q = sm + KktScratch::q; double* T = sm + KktScratch::T; double* f = sm + KktScratch::f;
    double* Kk = sm + KktScratch::K; double* kk = sm + KktScratch::kk; double* cf = sm + KktScratch::cf;
    // ---- terminal stage
    {
        const double* t = I.trec;
        for (int e = lane; e < NXA * NXA; e += KktLanes::n) {
            const int i = e % NXA, j = e / NXA;
            double v = t[T_H + e];
            if (i == j) v += dwreg + t[T_ZL + i] * t[T_IL + i] + t[T_ZU + i] * t[T_IU + i];
            P[e] = v;
        }
        for (int i = lane; i < NXA; i += KktLanes::n) p[i] = t[T_GN + i] - mu * t[T_IL + i] + mu * t[T_IU + i];
    }
#if MPCB_TERMCONS
    // Terminal equality E dx_N = -r_T with multiplier nu (new value solved for directly).  By linearity of the sweep
    // in the terminal gradient: p_k gains Pi_k nu, the feed-forward gains Gamma_k nu, and dx_N = h - G nu, with
    //   Pi_N = E',  Pi_k = (A_k + B_k K_k)' Pi_{k+1},  Gamma_k = -Muu^{-1} B_k' Pi_{k+1},
    //   G = sum_k (B_k' Pi_{k+1})' Muu^{-1} (B_k' Pi_{k+1}),   h = sum_k Pi_{k+1}' (B_k k_k + c_k)       (dx_0 = 0)
    // all accumulated in this same backward sweep; the caller then solves G nu = h + r_T.
    double* Pi = sm + KktScratch::PiA; double* Pn = sm + KktScratch::PiB;
    double* BtPi = sm + KktScratch::BtPi; double* Ga = sm + KktScratch::Ga;
    double* Gm = sm + KktScratch::Gm; double* hT = sm + KktScratch::hT;
    for (int e = lane; e < NXA * NXT; e += KktLanes::n) Pi[e] = (e % NXA == e / NXA) ? 1.0 : 0.0;
    for (int e = lane; e < NXT * NXT; e += KktLanes::n) Gm[e] = 0.0;
    for (int e = lane; e < NXT; e += KktLanes::n) hT[e] = 0.0;
#endif
    KktLanes::sync();
#if KKT_USE_TMA
    // the first KKT_NBUF - 1 records are requested up front, record k - (KKT_NBUF - 1) when stage k starts: the copies
    // stay that many stages ahead of the compute
    constexpr int AHEAD = KKT_NBUF - 1;
    if (lane == 0)
        for (int d = 0; d < AHEAD && NH - 1 - d >= 0; ++d)
            io.issue((NH - 1 - d) % KKT_NBUF, I.rec + (NH - 1 - d) * REC_SZ, KKT_RBUF, nullptr, 0);
#else
    (void)io;
#endif
    for (int k = NH - 1; k >= 0; --k) {
#if KKT_USE_TMA
        if (lane == 0 && k >= AHEAD) io.issue((k - AHEAD) % KKT_NBUF, I.rec + (k - AHEAD) * REC_SZ, KKT_RBUF, nullptr, 0);
        const double* R = io.wait(k % KKT_NBUF);
#else
        const double* R = I.rec + k * REC_SZ;          // one lane: the record is read in place
#endif
        double* fk = I.frec + k * FREC_SZ;
        // (a) P_{k+1}, p_{k+1} go to the forward record; slack coefficients
        for (int e = lane; e < NXA * NXA; e += KktLanes::n) fk[FREC_P + e] = P[e];
        for (int e = lane; e < NXA; e += KktLanes::n) fk[FREC_PV + e] = p[e];
#if MPCB_TERMCONS
        for (int e = lane; e < NXA * NXT; e += KktLanes::n) fk[FREC_PI + e] = Pi[e];
        for (int e = lane; e < NU * NXT; e += KktLanes::n) {
            const int l = e % NU, j = e / NU;
            double a = 0.0;
            for (int i = 0; i < NXA; ++i) a += R[R_AB + NXA * NXA + i + NXA * l] * Pi[i + NXA * j];
            BtPi[e] = a;
        }
#endif
#if NG > 0
        for (int r = lane; r < NG; r += KktLanes::n)
            cf[r] = (R[R_SG + r] + dwreg) * R[R_RG + r] - mu * R[R_ISL + r] + mu * R[R_ISU + r];
#endif
        // (b) f = P c + p ;  T = P [A B]
        for (int i = lane; i < NXA; i += KktLanes::n) {
            double a = p[i];
            for (int j = 0; j < NXA; ++j) a += P[i + NXA * j] * R[R_C + j];
            f[i] = a;
        }
        for (int e = lane; e < NXA * NZA; e += KktLanes::n) {
            const int i = e % NXA, j = e / NXA;
            double a = 0.0;
            for (int l = 0; l < NXA; ++l) a += P[i + NXA * l] * R[R_AB + l + NXA * j];
            T[e] = a;
        }
        KktLanes::sync();
        // (c) M = M0 + dw (I + G'G) + [A B]' P [A B] ;  q = grad - mu/dL + mu/dU + G' cf + [A B]' f
        for (int e = lane; e < NZA * NZA; e += KktLanes::n) {
            const int i = e % NZA, j = e / NZA;
            double m = R[R_M + e] + (i == j ? dwreg : 0.0);
#if NG > 0
            if (dwreg != 0.0) for (int r = 0; r < NG; ++r) m += dwreg * R[R_G + r + NG * i] * R[R_G + r + NG * j];
#endif
            for (int l = 0; l < NXA; ++l) m += R[R_AB + l + NXA * i] * T[l + NXA * j];
            M[e] = m;
        }
        for (int i = lane; i < NZA; i += KktLanes::n) {
            double a = R[R_GL + i] - mu * R[R_IL + i] + mu * R[R_IU + i];
#if NG > 0
            for (int r = 0; r < NG; ++r) a += R[R_G + r + NG * i] * cf[r];
#endif
            for (int l = 0; l < NXA; ++l) a += R[R_AB + l + NXA * i] * f[l];
            q[i] = a;
        }
        KktLanes::sync();
        // (d) Cholesky of the input block M_uu = L L' (every lane, in registers); Li = 1 / diag(L)
        double L[NU * NU], Li[NU];
        bool pd = true;
        for (int j = 0; j < NU; ++j) {
            double djj = M[(NXA + j) + NZA * (NXA + j)];
            for (int l = 0; l < j; ++l) djj -= L[j + NU * l] * L[j + NU * l];
            if (!(djj > 0.0)) { pd = false; djj = 1.0; }
#ifdef __CUDA_ARCH__
            const double inv = rsqrt(djj);
#else
            const double inv = 1.0 / sqrt(djj);
#endif
            Li[j] = inv;
            L[j + NU * j] = djj * inv;
            for (int i = j + 1; i < NU; ++i) {
                double a = M[(NXA + i) + NZA * (NXA + j)];
                for (int l = 0; l < j; ++l) a -= L[i + NU * l] * L[j + NU * l];
                L[i + NU * j] = a * inv;
            }
        }
        if (!pd) {                                               // uniform across the lanes
#if KKT_USE_TMA
            for (int d = 1; d <= KKT_NBUF - 1; ++d)              // drain the copies in flight before the sweep is repeated
                if (k >= d) io.wait((k - d) % KKT_NBUF);
            KktLanes::sync();
#endif
            return false;
        }
        // (e) K = -Muu^{-1} Mux (NU x NXA), kff = -Muu^{-1} q_u : one column per lane
        for (int c = lane; c <= NXA + NXT; c += KktLanes::n) {
            double y[NU];
            for (int i = 0; i < NU; ++i) {
#if MPCB_TERMCONS
                double a = (c < NXA) ? M[(NXA + i) + NZA * c] : ((c == NXA) ? q[NXA + i] : BtPi[i + NU * (c - NXA - 1)]);
#else
                double a = (c < NXA) ? M[(NXA + i) + NZA * c] : q[NXA + i];
#endif
                for (int l = 0; l < i; ++l) a -= L[i + NU * l] * y[l];
                y[i] = a * Li[i];
            }
            for (int i = NU - 1; i >= 0; --i) {
                double a = y[i];
                for (int l = i + 1; l < NU; ++l) a -= L[l + NU * i] * y[l];
                y[i] = a * Li[i];
            }
            for (int i = 0; i < NU; ++i) {
                if (c < NXA) { Kk[i + NU * c] = -y[i]; fk[FREC_K + i + NU * c] = -y[i]; }
                else if (c == NXA) { kk[i] = -y[i]; fk[FREC_KF + i] = -y[i]; }
#if MPCB_TERMCONS
                else { Ga[i + NU * (c - NXA - 1)] = -y[i]; fk[FREC_GA + i + NU * (c - NXA - 1)] = -y[i]; }
#endif
            }
        }
        KktLanes::sync();
#if MPCB_TERMCONS
        for (int e = lane; e < NXA * NXT; e += KktLanes::n) {
            const int i = e % NXA, j = e / NXA;
            double a = 0.0;
            for (int l = 0; l < NXA; ++l) a += R[R_AB + l + NXA * i] * Pi[l + NXA * j];
            for (int m = 0; m < NU; ++m) a += Kk[m + NU * i] * BtPi[m + NU * j];
            Pn[e] = a;
        }
        for (int e = lane; e < NXT * NXT; e += KktLanes::n) {
            const int j1 = e % NXT, j2 = e / NXT;
            double a = Gm[e];
            for (int m = 0; m < NU; ++m) a -= BtPi[m + NU * j1] * Ga[m + NU * j2];
            Gm[e] = a;
        }
        for (int j = lane; j < NXT; j += KktLanes::n) {
            double a = hT[j];
            for (int i = 0; i < NXA; ++i) {
                double bc = R[R_C + i];
                for (int m = 0; m < NU; ++m) bc += R[R_AB + NXA * NXA + i + NXA * m] * kk[m];
                a += Pi[i + NXA * j] * bc;
            }
            hT[j] = a;
        }
        { double* tmp = Pi; Pi = Pn; Pn = tmp; }
#endif
        // (f) P = Mxx + Mxu K (symmetrised), p = q_x + Mxu kff
        for (int e = lane; e < NXA * NXA; e += KktLanes::n) {
            const int i = e % NXA, j = e / NXA;
            double a = M[i + NZA * j], b = M[j + NZA * i];
            for (int l = 0; l < NU; ++l) { a += M[i + NZA * (NXA + l)] * Kk[l + NU * j]; b += M[j + NZA * (NXA + l)] * Kk[l + NU * i]; }
            P[e] = (i == j) ? a : 0.5 * (a + b);
        }
        for (int i = lane; i < NXA; i += KktLanes::n) {
            double a = q[i];
            for (int l = 0; l < NU; ++l) a += M[i + NZA * (NXA + l)] * kk[l];
            p[i] = a;
        }
        KktLanes::sync();
    }
    return true;
}

// end the solve of the instance run by the lane group G (ocp_kkt: KktLanes, ocp_accept: WarpLanes)
template <class G>
MPCB_HD void ocp_finish(OcpInst& I, const OcpShared& S, int status, double fval) {
    InstState& st = *I.st;
    if (S.o.honor_original_bounds)
        for (int i = NXA + G::id(); i < NWI; i += G::n) I.w[i] = fmin(fmax(I.w[i], S.lbx[i]), S.ubx[i]);
    if (G::id() == 0) { st.status = status; st.state = ST_DONE; st.fval = fval; }
    G::sync();
}

// Step-size bookkeeping for one bounded quantity with step dv, division free:
//   primal fraction to the boundary  alpha <= tau (v-lo)/(-dv)   <=>  alpha <= tau / max(-iL dv, iU dv)
//   dual   fraction to the boundary  alpha <= tau zL/(-dzL)      <=>  alpha <= tau / max(1 + iL dv - mu qL, 1 - iU dv - mu qU)
//   (dzL = mu iL - zL - zL iL dv,  qL = iL / zL), and the barrier part of the directional derivative.
MPCB_HD void step_terms(double dv, double iL, double iU, double qL, double qU, double mu,
                        double* rp, double* rd, double* gphid) {
    if (iL > 0.0) { *gphid -= mu * iL * dv; *rp = fmax(*rp, -iL * dv); *rd = fmax(*rd, 1.0 + iL * dv - mu * qL); }
    if (iU > 0.0) { *gphid += mu * iU * dv; *rp = fmax(*rp, iU * dv); *rd = fmax(*rd, 1.0 - iU * dv - mu * qU); }
}

// =============================================================================================
// kkt: one interior-point iteration up to (not including) the line search, for one instance
// =============================================================================================
MPCB_HD void ocp_kkt(OcpInst& I, const OcpShared& S, double* sm) {
    InstState& st = *I.st;
    const double rf = S.o.bound_relax;
    const int lane = KktLanes::id();
    const int iter = st.iter;
    // ---- reduce the per-stage partials written by the evaluation
    double fobj = 0.0, theta = 0.0, dual = 0.0, prim = 0.0, ysum = 0.0, zsum = 0.0, nbd = 0.0, pmin = 1e300, pmax = -1e300;
    double barr = 0.0;
    for (int k = lane; k <= NH; k += KktLanes::n) {
        const double* pp = (k < NH) ? (I.rec + k * REC_SZ + R_PART) : (I.trec + T_PART);
        fobj += pp[0]; theta += pp[1]; dual = fmax(dual, pp[2]); prim = fmax(prim, pp[3]); ysum += pp[4];
        zsum += pp[5]; nbd += pp[6]; pmin = fmin(pmin, pp[7]); pmax = fmax(pmax, pp[8]); barr += pp[9];
    }
    fobj = KktLanes::sum(fobj); theta = KktLanes::sum(theta); dual = KktLanes::max(dual); prim = KktLanes::max(prim); ysum = KktLanes::sum(ysum);
    zsum = KktLanes::sum(zsum); nbd = KktLanes::sum(nbd); pmin = KktLanes::min(pmin); pmax = KktLanes::max(pmax); barr = KktLanes::sum(barr);
#if NG > 0
    // A stage-0 range row that does not depend on u_0 is a constant (x_0 is fixed).  Outside its relaxed
    // bounds the OCP is infeasible: IPOPT would end in restoration with Infeasible_Problem_Detected, the
    // one status the reference loop reacts to (MPC_code.py:786,804; quirk D7 of SURVEY.md).
    if (iter == 0) {
        bool infeasible = false;
        const double* r0 = I.rec;
        for (int r = 0; r < NG; ++r) {
            bool constant = true;
            for (int j = NXA; j < NZA; ++j) if (r0[R_G + r + NG * j] != 0.0) constant = false;
            if (!constant) continue;
            const double v = r0[R_GV + r], lo = S.lbg[r], hi = S.ubg[r];
            if ((fin(lo) && v < rlo(lo, rf) - S.o.tol) || (fin(hi) && v > rhi(hi, rf) + S.o.tol)) infeasible = true;
        }
        if (infeasible) { ocp_finish<KktLanes>(I, S, 2, fobj); return; }
    }
#endif
    // ---- optimality error and termination (IPOPT: tol, dual_inf_tol=1, constr_viol_tol=1e-4, compl_inf_tol=1e-4)
    const double smax = 100.0;
    const double mc = (double)(NH * NXA + NH * NG + NXT);
    const double sd = fmax(smax, (ysum + zsum) / fmax(mc + nbd, 1.0)) / smax;
    const double sc = fmax(smax, zsum / fmax(nbd, 1.0)) / smax;
    const bool bounded = pmax >= pmin;
    const double c0 = bounded ? fmax(fabs(pmax), fabs(pmin)) : 0.0;
    const double E0 = fmax(fmax(dual / sd, prim), c0 / sc);
    int acc_cnt = st.acc_cnt;
    const bool resto = st.resto != 0;     // restoration iteration: no termination test, no barrier update (see ocp_accept)
    KktLanes::sync();
    if (lane == 0) st.E0 = E0;
    if (!(E0 == E0) || !fin(E0)) { ocp_finish<KktLanes>(I, S, -13, fobj); return; }
    if (!resto) {
        if (E0 <= S.o.tol && dual <= 1.0 && prim <= 1e-4 && c0 <= 1e-4) { ocp_finish<KktLanes>(I, S, 0, fobj); return; }
        if (E0 <= S.o.acceptable_tol && dual <= 1e10 && prim <= 1e-2 && c0 <= 1e-2) {
            acc_cnt += 1;
            if (acc_cnt >= S.o.acceptable_iter) { ocp_finish<KktLanes>(I, S, 1, fobj); return; }
        } else {
            acc_cnt = 0;
        }
    }
    if (iter >= S.o.max_iter) { ocp_finish<KktLanes>(I, S, -1, fobj); return; }
    // ---- monotone barrier update (kappa_eps=10, kappa_mu=0.2, theta_mu=1.5)
    double mu = st.mu;
    const double mu_min = S.o.tol / 10.0;
    bool changed = false;
    while (!resto && mu > mu_min) {
        const double cm = bounded ? fmax(fabs(pmax - mu), fabs(pmin - mu)) : 0.0;
        const double Emu = fmax(fmax(dual / sd, prim), cm / sc);
        if (Emu > 10.0 * mu) break;
        mu = fmax(mu_min, fmin(0.2 * mu, pow(mu, 1.5)));
        changed = true;
    }
    const double tau = changed ? fmax(0.99, 1.0 - mu) : st.tau;
    const double dw_last = st.dw_last;
    const double theta0_old = st.theta0;
    KktLanes::sync();
    // ---- Newton step by Riccati recursion, inertia-correcting ladder on delta_w
    double dwreg = 0.0;
    bool first = true, ok = false;
    KktIo io;
#if KKT_USE_TMA
    io.init(sm, lane);
    KktLanes::sync();
#endif
    for (int attempt = 0; attempt < 60; ++attempt) {
        if (ocp_riccati(I, mu, dwreg, sm, io)) { ok = true; break; }
        KktLanes::sync();
        if (first) { dwreg = (dw_last == 0.0) ? 1e-4 : fmax(1e-20, dw_last / 3.0); first = false; }
        else dwreg *= (dw_last == 0.0) ? 100.0 : 8.0;
        if (dwreg > 1e40) break;
    }
    if (!ok) { ocp_finish<KktLanes>(I, S, -3, fobj); return; }
#if MPCB_TERMCONS
    // ---- multiplier of the terminal equality: G nu = h + r_T (G is the horizon's reachability Gramian weighted by
    //      Muu^{-1}: positive definite when x_s can be reached; otherwise IPOPT's jacobian_regularization delta_c)
    {
        const double* Gm = sm + KktScratch::Gm; const double* hT = sm + KktScratch::hT; double* nuS = sm + KktScratch::nuS;
        double L[NXT * NXT + 1], y[NXT + 1];
        bool pd = false;
        for (int attempt = 0; attempt < 2 && !pd; ++attempt) {
            const double dc = attempt ? 1e-8 * pow(mu, 0.25) : 0.0;
            pd = true;
            for (int j = 0; j < NXT; ++j) {
                double djj = 0.5 * (Gm[j + NXT * j] + Gm[j + NXT * j]) + dc;
                for (int l = 0; l < j; ++l) djj -= L[j + NXT * l] * L[j + NXT * l];
                if (!(djj > 0.0)) { pd = false; break; }
                djj = sqrt(djj);
                L[j + NXT * j] = djj;
                for (int i = j + 1; i < NXT; ++i) {
                    double a = 0.5 * (Gm[i + NXT * j] + Gm[j + NXT * i]);
                    for (int l = 0; l < j; ++l) a -= L[i + NXT * l] * L[j + NXT * l];
                    L[i + NXT * j] = a / djj;
                }
            }
        }
        if (!pd) { ocp_finish<KktLanes>(I, S, -3, fobj); return; }
        for (int i = 0; i < NXT; ++i) {
            double a = hT[i] + I.trec[T_RT + i];
            for (int l = 0; l < i; ++l) a -= L[i + NXT * l] * y[l];
            y[i] = a / L[i + NXT * i];
        }
        for (int i = NXT - 1; i >= 0; --i) {
            double a = y[i];
            for (int l = i + 1; l < NXT; ++l) a -= L[l + NXT * i] * y[l];
            y[i] = a / L[i + NXT * i];
        }
        KktLanes::sync();
        for (int i = lane; i < NXT; i += KktLanes::n) { nuS[i] = y[i]; I.nuTn[i] = y[i]; }
        KktLanes::sync();
    }
#endif
    // ---- forward sweep, sequential part: only  du_k = K_k dx_k + k_k  and  dx_{k+1} = A dx_k + B du_k + c  (two lane
    //      phases per stage; the [A|B], c head of the record and the K, k head of the forward record come through the
    //      ring with lane groups and are read in place with one lane)
    double* dxa = sm + KktScratch::dx; double* du = sm + KktScratch::du; double* dxb = sm + KktScratch::dxn;
    for (int i = lane; i < NXA; i += KktLanes::n) { dxa[i] = 0.0; I.dw[i] = 0.0; }
#if KKT_USE_TMA
    // [A|B], c head of the record and K, k head of the forward record of stage k: two bulk copies into one ring buffer,
    // requested two stages ahead.  The forward records were written by this warp's ordinary stores in the backward sweep:
    // make them visible to the asynchronous proxy first.
    constexpr int NHEAD = (R_C + NXA + 1) / 2 * 2, NFH = (FREC_P + 1) / 2 * 2;
    static_assert(NHEAD + NFH <= KKT_RBUF, "forward heads must fit a ring buffer");
    asm volatile("fence.proxy.async;" ::: "memory");
    KktLanes::sync();
    if (lane == 0)
        for (int d = 0; d < KKT_NBUF - 1 && d < NH; ++d)
            io.issue(d % KKT_NBUF, I.rec + d * REC_SZ, NHEAD, I.frec + d * FREC_SZ, NFH);
#endif
    KktLanes::sync();
    for (int k = 0; k < NH; ++k) {
        double* dx = (k & 1) ? dxb : dxa; double* dxn = (k & 1) ? dxa : dxb;
#if KKT_USE_TMA
        if (lane == 0 && k + KKT_NBUF - 1 < NH)
            io.issue((k + KKT_NBUF - 1) % KKT_NBUF, I.rec + (k + KKT_NBUF - 1) * REC_SZ, NHEAD, I.frec + (k + KKT_NBUF - 1) * FREC_SZ, NFH);
        const double* R = io.wait(k % KKT_NBUF); const double* F = R + NHEAD;
#else
        const double* R = I.rec + k * REC_SZ; const double* F = I.frec + k * FREC_SZ;
#endif
        for (int i = lane; i < NU; i += KktLanes::n) {
            double a = F[FREC_KF + i];
            for (int j = 0; j < NXA; ++j) a += F[FREC_K + i + NU * j] * dx[j];
#if MPCB_TERMCONS
            for (int j = 0; j < NXT; ++j) a += F[FREC_GA + i + NU * j] * sm[KktScratch::nuS + j];
#endif
            du[i] = a;
            I.dw[k * NZA + NXA + i] = a;
        }
        KktLanes::sync();
        for (int i = lane; i < NXA; i += KktLanes::n) {
            double a = R[R_C + i];
            for (int j = 0; j < NXA; ++j) a += R[R_AB + i + NXA * j] * dx[j];
            for (int j = 0; j < NU; ++j) a += R[R_AB + NXA * NXA + i + NXA * j] * du[j];
            dxn[i] = a;
            I.dw[(k + 1) * NZA + i] = a;
        }
        KktLanes::sync();
    }
    // ---- stage-parallel part (lanes over stages): new dynamics multipliers, slack / multiplier steps of the range
    //      rows, fraction to the boundary (primal and dual) and the directional derivative of the barrier function
    double rp = 0.0, rd = 0.0, gphid = 0.0;       // largest primal / dual boundary ratios, directional derivative
    for (int k = lane; k <= NH; k += KktLanes::n) {
        if (k == NH) {
            const double* t = I.trec;
            for (int j = 0; j < NXA; ++j) {
                const double dv = I.dw[NH * NZA + j];
                gphid += t[T_GN + j] * dv;
                step_terms(dv, t[T_IL + j], t[T_IU + j], t[T_QL + j], t[T_QU + j], mu, &rp, &rd, &gphid);
            }
            continue;
        }
        const double* R = I.rec + k * REC_SZ; const double* F = I.frec + k * FREC_SZ;
        const double* dv = I.dw + k * NZA; const double* dxn = I.dw + (k + 1) * NZA;
        for (int i = 0; i < NXA; ++i) {
            double a = F[FREC_PV + i];
            for (int j = 0; j < NXA; ++j) a += F[FREC_P + i + NXA * j] * dxn[j];
#if MPCB_TERMCONS
            for (int j = 0; j < NXT; ++j) a += F[FREC_PI + i + NXA * j] * sm[KktScratch::nuS + j];
#endif
            I.lamn[k * NXA + i] = a;
        }
        for (int j = 0; j < NZA; ++j) {
            gphid += R[R_GL + j] * dv[j];
            step_terms(dv[j], R[R_IL + j], R[R_IU + j], R[R_QL + j], R[R_QU + j], mu, &rp, &rd, &gphid);
        }
#if NG > 0
        for (int r = 0; r < NG; ++r) {
            double dsr = R[R_RG + r];
            for (int j = 0; j < NZA; ++j) dsr += R[R_G + r + NG * j] * dv[j];
            const double b = -mu * R[R_ISL + r] + mu * R[R_ISU + r];
            I.ds[k * NG + r] = dsr;
            I.dym[k * NG + r] = (R[R_SG + r] + dwreg) * dsr + b - R[R_YM + r];
            step_terms(dsr, R[R_ISL + r], R[R_ISU + r], R[R_QSL + r], R[R_QSU + r], mu, &rp, &rd, &gphid);
        }
#endif
    }
    rp = KktLanes::max(rp); rd = KktLanes::max(rd); gphid = KktLanes::sum(gphid);
    const double amax = (rp > tau) ? tau / rp : 1.0;
    const double az = (rd > tau) ? tau / rd : 1.0;
    const double phi = fobj - mu * barr;
    const double theta0 = (theta0_old < 0.0) ? theta : theta0_old;
    const double theta_min = 1e-4 * fmax(1.0, theta0);
    // minimal step size before the line search gives up (gamma_alpha=0.05, gamma_theta=1e-5, gamma_phi=1e-8)
    double amin;
    if (gphid < 0.0 && theta <= theta_min) {
        amin = fmin(1e-5, fmin(1e-8 * theta / (-gphid), pow(theta, 1.1) / pow(-gphid, 2.3)));
    } else if (gphid < 0.0) {
        amin = fmin(1e-5, 1e-8 * theta / (-gphid));
    } else {
        amin = 1e-5;
    }
    if (lane == 0) {
        st.acc_cnt = acc_cnt;
        if (changed) { st.mu = mu; st.tau = tau; st.nfilt = 0; }
        if (dwreg > 0.0) st.dw_last = dwreg;
        st.theta0 = theta0;
        st.amin = 0.05 * amin;
        st.theta = theta; st.phi = phi; st.gphid = gphid; st.fval = fobj;
        st.alpha = amax; st.alpha_z = az;
        st.ls_iter = 0;
        st.state = ST_LS;
    }
    KktLanes::sync();
}

// =============================================================================================
// trial: constraint violation, objective and barrier terms of stage k at w + alpha dw
// =============================================================================================
MPCB_HD void ocp_trial_stage(OcpInst& I, const OcpShared& S, int k) {
    const double al = I.st->alpha, rf = S.o.bound_relax;
    const double* w = I.w; const double* dw = I.dw;
    double z[NXA], u[NU], d[ND + 1], px[NPX + 1], py[NPY + 1], t0, xn[NXA];
MPCB_UNROLL
    for (int i = 0; i < NXA; ++i) z[i] = w[k * NZA + i] + al * dw[k * NZA + i];
MPCB_UNROLL
    for (int i = 0; i < NU; ++i) u[i] = w[k * NZA + NXA + i] + al * dw[k * NZA + NXA + i];
    stage_params(I.par, k, d, px, py, &t0);
    double th = 0.0, prod = 1.0, l;     // prod: product of slacks-to-bounds (one log per stage)
#if MPCB_CONTFORM
    {
        ContCtx cc; cc.u = u; cc.par = I.par; cc.pxk = px; cc.pyk = py;
        double xt[NX + 1], xe[NX + 1];
MPCB_UNROLL
        for (int i = 0; i < NX; ++i) xt[i] = z[i];
        xt[NX] = 0.0;
        rk4_value_t<SysCont>(xt, cc, t0, xe);
MPCB_UNROLL
        for (int i = 0; i < NX; ++i) xn[i] = xe[i];
        l = xe[NX];
    }
#else
    dyn_value(z, u, d, px, t0, xn);
MPCB_UNROLL
    for (int i = NX; i < NXA; ++i) xn[i] = u[i - NX];
    ocp_cost(z, u, I.par, px, py, &l);
#endif
MPCB_UNROLL
    for (int i = 0; i < NXA; ++i) th += fabs(xn[i] - (w[(k + 1) * NZA + i] + al * dw[(k + 1) * NZA + i]));
#if NG > 0
    {
        double Y[NG];
        ocp_out(z, u, I.par, px, py, Y);
        for (int i = 0; i < NG; ++i) {
            const int gi = k * NG + i;
            const double st_ = I.s[gi] + al * I.ds[gi];
            th += fabs(Y[i] - st_);
            const double lo = S.lbg[gi], hi = S.ubg[gi];
            if (fin(lo)) prod *= st_ - rlo(lo, rf);
            if (fin(hi)) prod *= rhi(hi, rf) - st_;
        }
    }
#endif
    for (int j = (k == 0 ? NXA : 0); j < NZA; ++j) {
        const int wi = k * NZA + j;
        const double v = (j < NXA) ? z[j] : u[j - NXA];
        const double lo = S.lbx[wi], hi = S.ubx[wi];
        if (fin(lo)) prod *= v - rlo(lo, rf);
        if (fin(hi)) prod *= rhi(hi, rf) - v;
    }
    I.partt[k * 4 + 0] = l; I.partt[k * 4 + 1] = th; I.partt[k * 4 + 2] = log(prod);
    if (k == NH - 1) {
        double xN[NXA], V, pN = 1.0;
        for (int j = 0; j < NXA; ++j) {
            const int wi = NH * NZA + j;
            xN[j] = w[wi] + al * dw[wi];
            const double lo = S.lbx[wi], hi = S.ubx[wi];
            if (fin(lo)) pN *= xN[j] - rlo(lo, rf);
            if (fin(hi)) pN *= rhi(hi, rf) - xN[j];
        }
        ocp_term(xN, I.par, &V);
        double thT = 0.0;
#if MPCB_TERMCONS
        {
            double rT[NX];
            ocp_termc(xN, I.par, rT);
            for (int j = 0; j < NX; ++j) thT += fabs(rT[j]);
        }
#endif
        I.partt[NH * 4 + 0] = V; I.partt[NH * 4 + 1] = thT; I.partt[NH * 4 + 2] = log(pN);
    }
}

// =============================================================================================
// accept: filter line-search decision for one instance.  Always one warp per instance on the device
// (the updates are element-wise over w, lam, s, z), one lane on the host.
// =============================================================================================
MPCB_HD void ocp_accept(OcpInst& I, const OcpShared& S) {
    InstState& st = *I.st;
    const int lane = WarpLanes::id();
    const double rf = S.o.bound_relax, mu = st.mu;
    double th_t = 0.0, f_t = 0.0, b_t = 0.0;
    for (int k = lane; k <= NH; k += WarpLanes::n) { f_t += I.partt[k * 4 + 0]; th_t += I.partt[k * 4 + 1]; b_t += I.partt[k * 4 + 2]; }
    th_t = WarpLanes::sum(th_t); f_t = WarpLanes::sum(f_t); b_t = WarpLanes::sum(b_t);
    const double ph_t = f_t - mu * b_t;
    const double theta = st.theta, phi = st.phi, gphid = st.gphid, alpha = st.alpha, az = st.alpha_z;
    const double theta_min = 1e-4 * fmax(1.0, st.theta0), theta_max = 1e4 * fmax(1.0, st.theta0);
    const int nfilt = st.nfilt;
    bool ok = (th_t == th_t) && (ph_t == ph_t) && fin(th_t) && fin(ph_t) && th_t <= theta_max;
    if (ok)
        for (int i = 0; i < nfilt; ++i)
            if (th_t >= st.filt[2 * i] && ph_t >= st.filt[2 * i + 1]) { ok = false; break; }
    bool accepted = false, ftype = false;
    if (ok) {
        const bool switching = gphid < 0.0 && theta <= theta_min && alpha * pow(-gphid, 2.3) > pow(theta, 1.1);
        const double eps = 10.0 * 2.220446049250313e-16 * fabs(phi);
        if (switching) {
            if (ph_t - phi - eps <= 1e-8 * alpha * gphid) { accepted = true; ftype = true; }
        } else {
            if (th_t <= (1.0 - 1e-5) * theta || ph_t - eps <= phi - 1e-8 * theta) accepted = true;
        }
    }
    const double amin = st.amin;
    const int resto = st.resto, resto_calls = st.resto_calls;
    const double theta_entry = st.theta_entry;
    WarpLanes::sync();
    if (resto) {
        // ---- restoration iteration (proximal Gauss-Newton step on the constraint violation, see ocp_eval_stage):
        //      Armijo backtracking on the violation alone; multipliers restart from zero / mu over the slack; back to
        //      the regular iterations once the violation is kappa_resto = 0.9 of its value at entry and the filter
        //      (which holds the entry point) accepts the new point
        // a step shorter than 1e-5 of the Gauss-Newton step (jammed against the bounds, or no descent): the violation
        // cannot be reduced - a stationary point of the infeasibility (IPOPT: Infeasible_Problem_Detected)
        if (!(alpha > 1e-5)) { ocp_finish<WarpLanes>(I, S, theta > 1e-4 ? 2 : -2, st.fval); return; }
        const bool fine = (th_t == th_t) && fin(th_t) && th_t <= (1.0 - 1e-4 * alpha) * theta;
        if (!fine) {
            if (lane == 0) { st.alpha = 0.5 * alpha; st.ls_iter += 1; }
            WarpLanes::sync();
            return;
        }
        for (int i = NXA + lane; i < NWI; i += WarpLanes::n) {
            const double lo = S.lbx[i], hi = S.ubx[i];
            const double wn = I.w[i] + alpha * I.dw[i];
            if (fin(lo)) I.zL[i] = mu / (wn - rlo(lo, rf));
            if (fin(hi)) I.zU[i] = mu / (rhi(hi, rf) - wn);
            I.w[i] = wn;
        }
        for (int i = lane; i < NH * NXA; i += WarpLanes::n) I.lam[i] = 0.0;
        for (int i = lane; i < NXT; i += WarpLanes::n) I.nuT[i] = 0.0;
#if NG > 0
        for (int i = lane; i < NH * NG; i += WarpLanes::n) {
            const double lo = S.lbg[i], hi = S.ubg[i];
            const double sn = I.s[i] + alpha * I.ds[i];
            if (fin(lo)) I.vL[i] = mu / (sn - rlo(lo, rf));
            if (fin(hi)) I.vU[i] = mu / (rhi(hi, rf) - sn);
            I.s[i] = sn;
            I.ym[i] = 0.0;
        }
#endif
        bool leave = th_t <= 0.9 * theta_entry;
        if (leave)
            for (int i = 0; i < nfilt; ++i)
                if (th_t >= st.filt[2 * i] && ph_t >= st.filt[2 * i + 1]) { leave = false; break; }
        if (lane == 0) { st.iter += 1; st.state = ST_EVAL; if (leave) st.resto = 0; }
        WarpLanes::sync();
        return;
    }
    if (!accepted) {
        const double an = 0.5 * alpha;
        const bool give_up = !(an >= amin * (1.0 - 1e-12)) || an <= 1e-16;
        if (lane == 0) { st.alpha = an; st.ls_iter += 1; }
        WarpLanes::sync();
        if (give_up) {
            // IPOPT enters its restoration phase here: it looks for a point whose violation is kappa_resto times the
            // current one and which the filter, augmented by the current point, accepts; it reports
            // Infeasible_Problem_Detected (the status the reference loop acts on, MPC_code.py:786) when it ends at a
            // stationary point of the violation, and Restoration_Failed when called at an (almost) feasible point.
            // Same entry, goal and exits here; the sub-solver is simpler (proximal Gauss-Newton instead of an l1 IPM).
            if (theta < 1e-6 || resto_calls >= 3) { ocp_finish<WarpLanes>(I, S, theta > 1e-4 ? 2 : -2, st.fval); return; }
            if (lane == 0) {
                if (nfilt < MPCB_MAXFILT) {
                    st.filt[2 * nfilt] = (1.0 - 1e-5) * theta; st.filt[2 * nfilt + 1] = phi - 1e-8 * theta; st.nfilt = nfilt + 1;
                }
                st.resto = 1; st.resto_calls = resto_calls + 1; st.theta_entry = theta; st.state = ST_EVAL;
            }
            WarpLanes::sync();
        }
        return;
    }
    // ---- take the step; bound multipliers with their own step size, then the kappa_sigma safeguard
    const double ks = 1e10;
    for (int i = NXA + lane; i < NWI; i += WarpLanes::n) {
        const double lo = S.lbx[i], hi = S.ubx[i], dv = I.dw[i];
        const double wn = I.w[i] + alpha * dv;
        if (fin(lo)) {
            const double dl = I.w[i] - rlo(lo, rf), dln = wn - rlo(lo, rf);
            double z = I.zL[i] + az * (mu / dl - I.zL[i] - I.zL[i] / dl * dv);
            I.zL[i] = fmax(fmin(z, ks * mu / dln), mu / (ks * dln));
        }
        if (fin(hi)) {
            const double du = rhi(hi, rf) - I.w[i], dun = rhi(hi, rf) - wn;
            double z = I.zU[i] + az * (mu / du - I.zU[i] + I.zU[i] / du * dv);
            I.zU[i] = fmax(fmin(z, ks * mu / dun), mu / (ks * dun));
        }
        I.w[i] = wn;
    }
    for (int i = lane; i < NH * NXA; i += WarpLanes::n) I.lam[i] += alpha * (I.lamn[i] - I.lam[i]);
    for (int i = lane; i < NXT; i += WarpLanes::n) I.nuT[i] += alpha * (I.nuTn[i] - I.nuT[i]);
#if NG > 0
    for (int i = lane; i < NH * NG; i += WarpLanes::n) {
        const double lo = S.lbg[i], hi = S.ubg[i], dv = I.ds[i];
        const double sn = I.s[i] + alpha * dv;
        if (fin(lo)) {
            const double dl = I.s[i] - rlo(lo, rf), dln = sn - rlo(lo, rf);
            double z = I.vL[i] + az * (mu / dl - I.vL[i] - I.vL[i] / dl * dv);
            I.vL[i] = fmax(fmin(z, ks * mu / dln), mu / (ks * dln));
        }
        if (fin(hi)) {
            const double du = rhi(hi, rf) - I.s[i], dun = rhi(hi, rf) - sn;
            double z = I.vU[i] + az * (mu / du - I.vU[i] + I.vU[i] / du * dv);
            I.vU[i] = fmax(fmin(z, ks * mu / dun), mu / (ks * dun));
        }
        I.s[i] = sn;
        I.ym[i] += alpha * I.dym[i];
    }
#endif
    if (lane == 0) {
        if (!ftype && nfilt < MPCB_MAXFILT) {
            st.filt[2 * nfilt] = (1.0 - 1e-5) * theta;
            st.filt[2 * nfilt + 1] = phi - 1e-8 * theta;
            st.nfilt = nfilt + 1;
        }
        st.iter += 1;
        st.state = ST_EVAL;
    }
    WarpLanes::sync();
}
