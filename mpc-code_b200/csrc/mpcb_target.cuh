// mpcb_target.cuh - steady-state target problem, estimator update and plant maps (one thread per instance).
//
// Target: replaces `solver_ss(lbx,ubx,x0,p,lbg,ubg)` at MPC_code.py:704-709 for the NLP of
// Target_Calc.py:20-161 (variables [Xs,Us,Ys]; equalities Fx(Xs,Us)-Xs = 0 and
// Fy(Xs,Us)+lam(Us-Us_prev)-Ys = 0; box bounds), with the same interior-point algorithm as the OCP
// but a small dense KKT system factorised by Bunch-Kaufman LDL' (inertia from the pivots).
// Estimator: Estimator.py:231-386.  Plant: Utilities.py:21-100 as called at MPC_code.py:531-534,813-816.
#pragma once
#include "mpcb_ocp.cuh"
#ifndef MPCB_SENS_TGT
#define MPCB_SENS_TGT 0                   // 1: the generator wrote the target problem's mixed derivatives (tgt_*_dth)
#endif
#if MPCB_SENS_TGT
#include "mpcb_sens.cuh"                  // sens_dyn_dp: the d / px columns of the model equalities
#endif

#define NWS  MPCB_NWSS
// user rows of the target problem (Target_Calc.py:87-109): NGT inequalities g_SS <= 0, each with a slack variable
// s in (-inf, 0] (g - s = 0, the formulation of IPOPT and of oracle/ipm.py), NHT equalities h_SS = 0
#ifndef MPCB_NGSS
#define MPCB_NGSS 0
#endif
#ifndef MPCB_NHSS
#define MPCB_NHSS 0
#endif
#define NGT  MPCB_NGSS
#define NHT  MPCB_NHSS
#define NOUT (NY + NGT + NHT)          // rows of tgt_out: output map, g_SS, h_SS
#define NVT  (NWS + NGT)               // variables of the interior-point solve: [xs, us, ys, slacks]
#define MCS  (NX + NOUT)
#define NKS  (NVT + MCS)
#define NWSP (NWS * (NWS + 1) / 2)

// ---------------------------------------------------------------------------------------------
// dense symmetric indefinite factorisation (Bunch-Kaufman, lower, unblocked) and solve
// ---------------------------------------------------------------------------------------------
template <int N>
MPCB_HD void bk_factor(double* A, int* ipiv, int* npos, int* nneg, int* nzero) {
    const double alpha = (1.0 + sqrt(17.0)) / 8.0;
    *npos = *nneg = *nzero = 0;
    int k = 0;
    while (k < N) {
        int kstep = 1, kp = k;
        const double absakk = fabs(A[k + N * k]);
        int imax = k; double colmax = 0.0;
        for (int i = k + 1; i < N; ++i) { const double v = fabs(A[i + N * k]); if (v > colmax) { colmax = v; imax = i; } }
        if (fmax(absakk, colmax) == 0.0) {
            *nzero += 1; ipiv[k] = k + 1; k += 1; continue;
        }
        if (absakk >= alpha * colmax) {
            kp = k;
        } else {
            double rowmax = 0.0;
            for (int j = k; j < imax; ++j) rowmax = fmax(rowmax, fabs(A[imax + N * j]));
            for (int i = imax + 1; i < N; ++i) rowmax = fmax(rowmax, fabs(A[i + N * imax]));
            if (absakk >= alpha * colmax * (colmax / rowmax)) kp = k;
            else if (fabs(A[imax + N * imax]) >= alpha * rowmax) kp = imax;
            else { kp = imax; kstep = 2; }
        }
        const int kk = k + kstep - 1;
        if (kp != kk) {
            for (int i = kp + 1; i < N; ++i) { const double t = A[i + N * kk]; A[i + N * kk] = A[i + N * kp]; A[i + N * kp] = t; }
            for (int j = kk + 1; j < kp; ++j) { const double t = A[j + N * kk]; A[j + N * kk] = A[kp + N * j]; A[kp + N * j] = t; }
            { const double t = A[kk + N * kk]; A[kk + N * kk] = A[kp + N * kp]; A[kp + N * kp] = t; }
            if (kstep == 2) { const double t = A[k + 1 + N * k]; A[k + 1 + N * k] = A[kp + N * k]; A[kp + N * k] = t; }
        }
        if (kstep == 1) {
            const double dkk = A[k + N * k];
            if (dkk > 0.0) *npos += 1; else if (dkk < 0.0) *nneg += 1; else *nzero += 1;
            const double r1 = 1.0 / dkk;
            for (int j = k + 1; j < N; ++j) {
                const double ajk = A[j + N * k] * r1;
                for (int i = j; i < N; ++i) A[i + N * j] -= A[i + N * k] * ajk;
            }
            for (int i = k + 1; i < N; ++i) A[i + N * k] *= r1;
            ipiv[k] = kp + 1;
        } else {
            const double a = A[k + N * k], b = A[k + 1 + N * k], c = A[k + 1 + N * (k + 1)];
            const double det = a * c - b * b;
            if (det < 0.0) { *npos += 1; *nneg += 1; }
            else if (det > 0.0) { if (a + c > 0.0) *npos += 2; else *nneg += 2; }
            else *nzero += 1;
            if (k < N - 2) {
                double d21 = b;
                const double d11 = c / d21, d22 = a / d21;
                const double t = 1.0 / (d11 * d22 - 1.0);
                d21 = t / d21;
                for (int j = k + 2; j < N; ++j) {
                    const double wk = d21 * (d11 * A[j + N * k] - A[j + N * (k + 1)]);
                    const double wkp1 = d21 * (d22 * A[j + N * (k + 1)] - A[j + N * k]);
                    for (int i = j; i < N; ++i) A[i + N * j] -= A[i + N * k] * wk + A[i + N * (k + 1)] * wkp1;
                    A[j + N * k] = wk;
                    A[j + N * (k + 1)] = wkp1;
                }
            }
            ipiv[k] = -(kp + 1); ipiv[k + 1] = -(kp + 1);
        }
        k += kstep;
    }
}

template <int N>
MPCB_HD void bk_solve(const double* A, const int* ipiv, double* b) {
    int k = 0;
    while (k < N) {
        if (ipiv[k] > 0) {
            const int kp = ipiv[k] - 1;
            if (kp != k) { const double t = b[k]; b[k] = b[kp]; b[kp] = t; }
            for (int i = k + 1; i < N; ++i) b[i] -= b[k] * A[i + N * k];
            b[k] /= A[k + N * k];
            k += 1;
        } else {
            const int kp = -ipiv[k] - 1;
            if (kp != k + 1) { const double t = b[k + 1]; b[k + 1] = b[kp]; b[kp] = t; }
            for (int i = k + 2; i < N; ++i) b[i] -= b[k] * A[i + N * k] + b[k + 1] * A[i + N * (k + 1)];
            const double akm1k = A[k + 1 + N * k];
            const double akm1 = A[k + N * k] / akm1k, ak = A[k + 1 + N * (k + 1)] / akm1k;
            const double denom = akm1 * ak - 1.0;
            const double bkm1 = b[k] / akm1k, bk = b[k + 1] / akm1k;
            b[k] = (ak * bkm1 - bk) / denom;
            b[k + 1] = (akm1 * bk - bkm1) / denom;
            k += 2;
        }
    }
    k = N - 1;
    while (k >= 0) {
        if (ipiv[k] > 0) {
            double a = b[k];
            for (int i = k + 1; i < N; ++i) a -= A[i + N * k] * b[i];
            b[k] = a;
            const int kp = ipiv[k] - 1;
            if (kp != k) { const double t = b[k]; b[k] = b[kp]; b[kp] = t; }
            k -= 1;
        } else {
            double a = b[k], a1 = b[k - 1];
            for (int i = k + 1; i < N; ++i) { a -= A[i + N * k] * b[i]; a1 -= A[i + N * (k - 1)] * b[i]; }
            b[k] = a; b[k - 1] = a1;
            const int kp = -ipiv[k] - 1;
            if (kp != k) { const double t = b[k]; b[k] = b[kp]; b[kp] = t; }
            k -= 2;
        }
    }
}

#if MPCB_HAS_TARGET
struct TgtShared { const double *lbx, *ubx; IpmOpts o; };

// constraint values (and derivatives) of the target problem at v = [xs, us, ys, slacks]; rows [dyn | out | g_SS - s | h_SS]
MPCB_HD void tgt_eval(const double* w, const double* par, const double* lam, bool derivs,
                      double* f, double* c, double* grad, double* J /*MCS x NVT col-major*/, double* Hp /*NWSP*/) {
    const double* d = par + MPCB_OFFSS_D; const double* px = par + MPCB_OFFSS_PX;
    const double t0 = par[MPCB_OFFSS_T];
    double dl[ND + 1], pxl[NPX + 1];
    for (int i = 0; i < ND; ++i) dl[i] = d[i];
    for (int i = 0; i < NPX; ++i) pxl[i] = px[i];
    double xn[NX];
    if (!derivs) {
        dyn_value(w, w + NX, dl, pxl, t0, xn);
        for (int i = 0; i < NX; ++i) c[i] = xn[i] - w[i];
        tgt_out(w, par, c + NX);
        for (int i = 0; i < NGT; ++i) c[NX + NY + i] -= w[NWS + i];
        tgt_cost(w, par, f);
        return;
    }
    double A[NX * NX], Bm[NX * NU], Hd[NZP], Hc[NWSP], Ho[NWSP], Jo[NOUT * NWS];
    for (int i = 0; i < NZP; ++i) Hd[i] = 0.0;
    dyn_full(w, w + NX, dl, pxl, t0, lam, xn, A, Bm, Hd);
    for (int i = 0; i < NX; ++i) c[i] = xn[i] - w[i];
    tgt_out_d(w, par, lam + NX, c + NX, Jo, Ho);
    for (int i = 0; i < NGT; ++i) c[NX + NY + i] -= w[NWS + i];
    tgt_cost_d(w, par, f, grad, Hc);
    for (int i = 0; i < NGT; ++i) grad[NWS + i] = 0.0;
    for (int i = 0; i < NWSP; ++i) Hp[i] = Hc[i] + Ho[i];
    for (int i = 0; i < NZP; ++i) Hp[i] += Hd[i];            // (xs,us) block leads the packed triangle
    for (int j = 0; j < NWS; ++j) {
        for (int i = 0; i < NX; ++i) {
            double v = 0.0;
            if (j < NX) v = A[i + NX * j] - (i == j ? 1.0 : 0.0);
            else if (j < NZ) v = Bm[i + NX * (j - NX)];
            J[i + MCS * j] = v;
        }
        for (int i = 0; i < NOUT; ++i) J[NX + i + MCS * j] = Jo[i + NOUT * j];
    }
    for (int j = 0; j < NGT; ++j)                            // slack columns
        for (int i = 0; i < MCS; ++i) J[i + MCS * (NWS + j)] = (i == NX + NY + j) ? -1.0 : 0.0;
}

#if MPCB_SENS_TGT
// ---------------------------------------------------------------------------------------------
// Sensitivities of the target solution with respect to theta_ss = [usp | ysp | xsp | d | Us_prev | px | py] (par_ss
// without vec(lam) and t, which are held constant).  At the returned iterate the barrier KKT system F(v; theta_ss) = 0
// of v = [xs, us, ys, slacks] is differentiated: dv/dtheta_ss = -K^{-1} dF/dtheta_ss, with K the matrix of the Newton
// step (Hessian of the Lagrangian + Sigma = Z / D on the bounded variables, J and J') without regularisation, and
// dF/dtheta_ss = [d(grad_v L)/dtheta_ss ; dc/dtheta_ss] with the final equality multipliers.  The bounds are shared
// constants and add no theta terms.  With honor_original_bounds the solve clips w after its loop: the derivative is
// taken at the iterate before that clipping (the stored wss is the clipped one, which mpcb_target returns).
// The solve keeps its multipliers in registers, so the capture solves the problem again from the same guess, with the
// same code (tgt_solve_t<., true>), and builds the capture in the solver's tail.
// ---------------------------------------------------------------------------------------------
#define NTS MPCB_NTHSS
struct TgtSensLayout {                                               // doubles per instance
    static constexpr int head = 0;                                   // [0] status (0 / 1 / 2), [1] status of the solve
    static constexpr int w = 2;                                      // NWS  the solution (mpcb_target's output)
    static constexpr int K = w + NWS;                                // NKS*NKS  Bunch-Kaufman factor of K
    static constexpr int piv = K + NKS * NKS;                        // NKS  its pivots
    static constexpr int fth = piv + NKS;                            // NKS*NTS  dF/dtheta_ss, column-major
    static constexpr int total = (fth + NKS * NTS + 1) / 2 * 2;
};

// dF/dtheta_ss at (w, y), rows [grad_v L (NVT) | c (MCS)]; the slack rows and columns have no theta terms
MPCB_HD void tgt_eval_dth(const double* w, const double* par, const double* y, double* Fth) {
    double Lt[NWS * NTS], Yt[NOUT * NTS], HYt[NWS * NTS];
    tgt_cost_dth(w, par, Lt);
    tgt_out_dth(w, par, y + NX, Yt, HYt);
    for (int e = 0; e < NKS * NTS; ++e) Fth[e] = 0.0;
    for (int t = 0; t < NTS; ++t) {
        for (int j = 0; j < NWS; ++j) Fth[j + NKS * t] = Lt[j + NWS * t] + HYt[j + NWS * t];
        for (int i = 0; i < NOUT; ++i) Fth[NVT + NX + i + NKS * t] = Yt[i + NOUT * t];
    }
    // d and px enter the model equalities Fx(xs, us) - xs = 0 (theta_ss columns OFFSS_D + c and OFFSS_LAM + c - ND)
    double dl[ND + 1], pxl[NPX + 1], Fm[NX * NPM + 1], Hm[NZ * NPM + 1];
    for (int i = 0; i < ND; ++i) dl[i] = par[MPCB_OFFSS_D + i];
    for (int i = 0; i < NPX; ++i) pxl[i] = par[MPCB_OFFSS_PX + i];
    sens_dyn_dp(w, w + NX, dl, pxl, par[MPCB_OFFSS_T], y, Fm, Hm);
    for (int c = 0; c < NPM; ++c) {
        const int t = c < ND ? MPCB_OFFSS_D + c : MPCB_OFFSS_LAM + (c - ND);
        for (int r = 0; r < NZ; ++r) Fth[r + NKS * t] += Hm[r + NZ * c];
        for (int i = 0; i < NX; ++i) Fth[NVT + i + NKS * t] += Fm[i + NX * c];
    }
}

// Capture at the final iterate of a solve that ended with `status`: K without regularisation, its factor and inertia
// check (NVT, MCS, 0), dF/dtheta_ss.  cap[0]: 0 computed, 1 the solve ended with a status other than 0 / 1, 2 wrong inertia.
MPCB_HD void tgt_capture(const double* par, const double* w, const double* y, const double* zL, const double* zU,
                         const double* lo, const double* hi, const bool* hl, const bool* hu, const double* J,
                         const double* Hp, int status, double* cap) {
    cap[1] = (double)status;
    if (status != 0 && status != 1) { cap[TgtSensLayout::head] = 1.0; return; }
    double K[NKS * NKS]; int ipiv[NKS], np_, nn_, nz_;
    for (int i = 0; i < NKS * NKS; ++i) K[i] = 0.0;
    for (int j = 0; j < NVT; ++j) {
        if (j < NWS) for (int i = j; i < NWS; ++i) K[i + NKS * j] = Hp[tri(i, j)];
        double sig = 0.0;
        if (hl[j]) sig += zL[j] / (w[j] - lo[j]);
        if (hu[j]) sig += zU[j] / (hi[j] - w[j]);
        K[j + NKS * j] += sig;
        for (int i = 0; i < MCS; ++i) K[NVT + i + NKS * j] = J[i + MCS * j];
    }
    bk_factor<NKS>(K, ipiv, &np_, &nn_, &nz_);
    for (int i = 0; i < NKS * NKS; ++i) cap[TgtSensLayout::K + i] = K[i];
    for (int i = 0; i < NKS; ++i) cap[TgtSensLayout::piv + i] = (double)ipiv[i];
    tgt_eval_dth(w, par, y, cap + TgtSensLayout::fth);
    cap[TgtSensLayout::head] = (np_ == NVT && nn_ == MCS && nz_ == 0) ? 0.0 : 2.0;
}
#endif  // MPCB_SENS_TGT

// Whole interior-point solve of one target problem (same algorithm as oracle/ipm.py and mpcb_ocp.cuh).
// MPCB_TGT_RESTO = false: the regular iterations only; a failed line search returns TGT_NEEDS_RESTO and `tgt_solve`
// repeats the (cold-started, deterministic) solve with the variant that carries the feasibility restoration.  Keeping
// the restoration out of the common variant halves its register spills (ptxas: 520 / 1288 B vs 1132 / 1930 B).
// CAPTURE = true (mpcb_target_sens_factor): the tail also writes the sensitivity capture `cap` of the final iterate.
#define TGT_NEEDS_RESTO 1000
template <bool MPCB_TGT_RESTO, bool CAPTURE = false>
MPCB_HD void tgt_solve_t(const double* par, double* w_io, double* fout, int* status_out, int* iters_out, const TgtShared& S,
                         double* cap = nullptr) {
    const IpmOpts& o = S.o;
    const double rf = o.bound_relax;
    double w[NVT], lo[NVT], hi[NVT]; bool hl[NVT], hu[NVT];
    int nb = 0;
    for (int i = 0; i < NWS; ++i) {
        hl[i] = fin(S.lbx[i]); hu[i] = fin(S.ubx[i]);
        lo[i] = hl[i] ? rlo(S.lbx[i], rf) : S.lbx[i];
        hi[i] = hu[i] ? rhi(S.ubx[i], rf) : S.ubx[i];
        nb += (hl[i] ? 1 : 0) + (hu[i] ? 1 : 0);
        w[i] = push_in(w_io[i], lo[i], hi[i], o.bound_push);
    }
    if (NGT > 0) {                      // slacks start at g_SS(pushed point), pushed into (-inf, 0] (oracle/ipm.py: starting point)
        double f0, c0[MCS];
        for (int i = NWS; i < NVT; ++i) w[i] = 0.0;
        tgt_eval(w, par, nullptr, false, &f0, c0, nullptr, nullptr, nullptr);
        for (int i = NWS; i < NVT; ++i) {
            hl[i] = false; hu[i] = true; lo[i] = -INFINITY; hi[i] = rhi(0.0, rf); nb += 1;
            w[i] = push_in(c0[NX + NY + (i - NWS)], lo[i], hi[i], o.bound_push);
        }
    }
    double y[MCS], zL[NVT], zU[NVT];
    for (int i = 0; i < MCS; ++i) y[i] = 0.0;
    for (int i = 0; i < NVT; ++i) { zL[i] = hl[i] ? 1.0 : 0.0; zU[i] = hu[i] ? 1.0 : 0.0; }
    double mu = o.mu_init, tau = fmax(0.99, 1.0 - mu), dw_last = 0.0, theta0 = -1.0;
    double filt[2 * MPCB_MAXFILT]; int nfilt = 0, acc = 0, it = 0, status = -1;
    bool resto = false; int resto_calls = 0; double theta_entry = 0.0;      // feasibility restoration, as in ocp_accept
    double f = 0.0, c[MCS], grad[NVT], J[MCS * NVT], Hp[NWSP];
    bool evaluate = true;               // ONE call site of the derivative evaluation (three inlined RK4 sweeps): the solver's
    while (true) {                      // code is 240 kB otherwise and a sixth of its stalls are instruction fetches
        if (evaluate) tgt_eval(w, par, y, true, &f, c, grad, J, Hp);
        evaluate = false;
        if (it == 0 && !resto) {        // IPOPT: a starting point whose functions do not evaluate ends the solve with -13
            double chk = f;
            for (int i = 0; i < MCS; ++i) chk += c[i];
            for (int i = 0; i < NVT; ++i) chk += grad[i];
            if (!(chk == chk) || !fin(chk)) { status = -13; break; }
        }
        // optimality error
        double dual = 0.0, prim = 0.0, ysum = 0.0, zsum = 0.0, c0 = 0.0;
        for (int j = 0; j < NVT; ++j) {
            double r = grad[j] - zL[j] + zU[j];
            for (int i = 0; i < MCS; ++i) r += J[i + MCS * j] * y[i];
            dual = fmax(dual, fabs(r));
            zsum += zL[j] + zU[j];
            if (hl[j]) c0 = fmax(c0, fabs((w[j] - lo[j]) * zL[j]));
            if (hu[j]) c0 = fmax(c0, fabs((hi[j] - w[j]) * zU[j]));
        }
        for (int i = 0; i < MCS; ++i) { prim = fmax(prim, fabs(c[i])); ysum += fabs(y[i]); }
        const double sd = fmax(100.0, (ysum + zsum) / (double)(MCS + nb > 0 ? MCS + nb : 1)) / 100.0;
        const double sc = fmax(100.0, zsum / (double)(nb > 0 ? nb : 1)) / 100.0;
        const double E0 = fmax(fmax(dual / sd, prim), c0 / sc);
        if (!(E0 == E0) || !fin(E0)) { status = -13; break; }
        if (!resto) {
            if (E0 <= o.tol && dual <= 1.0 && prim <= 1e-4 && c0 <= 1e-4) { status = 0; break; }
            if (E0 <= o.acceptable_tol && dual <= 1e10 && prim <= 1e-2 && c0 <= 1e-2) {
                if (++acc >= o.acceptable_iter) { status = 1; break; }
            } else acc = 0;
        }
        if (it >= o.max_iter) { status = -1; break; }
        // barrier update
        const double mu_min = o.tol / 10.0;
        bool changed = false;
        while (!resto && mu > mu_min) {
            double cm = 0.0;
            for (int j = 0; j < NVT; ++j) {
                if (hl[j]) cm = fmax(cm, fabs((w[j] - lo[j]) * zL[j] - mu));
                if (hu[j]) cm = fmax(cm, fabs((hi[j] - w[j]) * zU[j] - mu));
            }
            if (fmax(fmax(dual / sd, prim), cm / sc) > 10.0 * mu) break;
            mu = fmax(mu_min, fmin(0.2 * mu, pow(mu, 1.5)));
            changed = true;
        }
        if (changed) { tau = fmax(0.99, 1.0 - mu); nfilt = 0; }
        // Newton system with inertia correction
        double K[NKS * NKS], rhs[NKS]; int ipiv[NKS];
        double dwreg = 0.0, dcreg = 0.0; bool first = true, ok = false;
        for (int attempt = 0; attempt < 60; ++attempt) {
            for (int i = 0; i < NKS * NKS; ++i) K[i] = 0.0;
            for (int j = 0; j < NVT; ++j) {
                if (j < NWS) for (int i = j; i < NWS; ++i) K[i + NKS * j] = resto ? 0.0 : Hp[tri(i, j)];
                double sig = dwreg;
                if (resto) {             // proximal Gauss-Newton step: zeta D_R^2 + primal barrier Hessian
                    const double sc = fmax(1.0, fabs(w[j]));
                    sig += sqrt(mu) / (sc * sc);
                    if (hl[j]) { const double d = w[j] - lo[j]; sig += mu / (d * d); }
                    if (hu[j]) { const double d = hi[j] - w[j]; sig += mu / (d * d); }
                } else {
                    if (hl[j]) sig += zL[j] / (w[j] - lo[j]);
                    if (hu[j]) sig += zU[j] / (hi[j] - w[j]);
                }
                K[j + NKS * j] += sig;
                for (int i = 0; i < MCS; ++i) K[NVT + i + NKS * j] = J[i + MCS * j];
            }
            for (int i = 0; i < MCS; ++i) K[NVT + i + NKS * (NVT + i)] = -dcreg;
            int np_, nn_, nz_;
            bk_factor<NKS>(K, ipiv, &np_, &nn_, &nz_);
            if (np_ == NVT && nn_ == MCS && nz_ == 0) { ok = true; break; }
            if (nz_ > 0) dcreg = 1e-8 * pow(mu, 0.25);
            if (first) { dwreg = (dw_last == 0.0) ? 1e-4 : fmax(1e-20, dw_last / 3.0); first = false; }
            else dwreg *= (dw_last == 0.0) ? 100.0 : 8.0;
            if (dwreg > 1e40) break;
        }
        if (!ok) { status = -3; break; }
        if (dwreg > 0.0) dw_last = dwreg;
        for (int j = 0; j < NVT; ++j) {
            double r = grad[j];
            for (int i = 0; i < MCS; ++i) r += J[i + MCS * j] * y[i];
            if (resto) r = 0.0;
            if (hl[j]) r -= mu / (w[j] - lo[j]);
            if (hu[j]) r += mu / (hi[j] - w[j]);
            rhs[j] = -r;
        }
        for (int i = 0; i < MCS; ++i) rhs[NVT + i] = -c[i];
        bk_solve<NKS>(K, ipiv, rhs);
        // step sizes, barrier objective
        double amax = 1.0, az = 1.0, gphid = 0.0, barr = 0.0, theta = 0.0;
        double dzL[NVT], dzU[NVT];
        for (int j = 0; j < NVT; ++j) {
            const double dv = rhs[j];
            gphid += grad[j] * dv;
            dzL[j] = dzU[j] = 0.0;
            if (hl[j]) {
                const double dl = w[j] - lo[j];
                barr += log(dl); gphid -= mu / dl * dv;
                if (dv < 0.0) amax = fmin(amax, -tau * dl / dv);
                dzL[j] = mu / dl - zL[j] - zL[j] / dl * dv;
                if (dzL[j] < 0.0) az = fmin(az, -tau * zL[j] / dzL[j]);
            }
            if (hu[j]) {
                const double du = hi[j] - w[j];
                barr += log(du); gphid += mu / du * dv;
                if (dv > 0.0) amax = fmin(amax, tau * du / dv);
                dzU[j] = mu / du - zU[j] + zU[j] / du * dv;
                if (dzU[j] < 0.0) az = fmin(az, -tau * zU[j] / dzU[j]);
            }
        }
        for (int i = 0; i < MCS; ++i) theta += fabs(c[i]);
        const double phi = f - mu * barr;
        if (theta0 < 0.0) theta0 = theta;
        const double theta_min = 1e-4 * fmax(1.0, theta0), theta_max = 1e4 * fmax(1.0, theta0);
        double amin;
        if (gphid < 0.0 && theta <= theta_min) amin = fmin(1e-5, fmin(1e-8 * theta / (-gphid), pow(theta, 1.1) / pow(-gphid, 2.3)));
        else if (gphid < 0.0) amin = fmin(1e-5, 1e-8 * theta / (-gphid));
        else amin = 1e-5;
        amin *= 0.05;
        double alpha = amax; bool accepted = false, ftype = false;
        double wt[NVT], ft, ct[MCS];
        if (MPCB_TGT_RESTO && resto) {  // restoration iteration: Armijo on the violation alone
            double th_t = 0.0;
            while (alpha > 1e-5) {         // shorter: jammed against the bounds / no descent -> the violation cannot be reduced
                for (int j = 0; j < NVT; ++j) wt[j] = w[j] + alpha * rhs[j];
                tgt_eval(wt, par, y, false, &ft, ct, nullptr, nullptr, nullptr);
                th_t = 0.0;
                for (int i = 0; i < MCS; ++i) th_t += fabs(ct[i]);
                if ((th_t == th_t) && fin(th_t) && th_t <= (1.0 - 1e-4 * alpha) * theta) { accepted = true; break; }
                alpha *= 0.5;
            }
            if (!accepted) { status = theta > 1e-4 ? 2 : -2; break; }
            double b_t = 0.0;
            for (int j = 0; j < NVT; ++j) {
                w[j] = wt[j];
                if (hl[j]) { const double d = w[j] - lo[j]; zL[j] = mu / d; b_t += log(d); }
                if (hu[j]) { const double d = hi[j] - w[j]; zU[j] = mu / d; b_t += log(d); }
            }
            for (int i = 0; i < MCS; ++i) y[i] = 0.0;
            const double ph_t = ft - mu * b_t;
            bool leave = th_t <= 0.9 * theta_entry;
            if (leave) for (int i = 0; i < nfilt; ++i) if (th_t >= filt[2 * i] && ph_t >= filt[2 * i + 1]) { leave = false; break; }
            if (leave) resto = false;
            it += 1;
            evaluate = true;
            continue;
        }
        while (alpha >= amin * (1.0 - 1e-12) && alpha > 1e-16) {
            for (int j = 0; j < NVT; ++j) wt[j] = w[j] + alpha * rhs[j];
            tgt_eval(wt, par, y, false, &ft, ct, nullptr, nullptr, nullptr);
            double th_t = 0.0, b_t = 0.0;
            for (int i = 0; i < MCS; ++i) th_t += fabs(ct[i]);
            for (int j = 0; j < NVT; ++j) { if (hl[j]) b_t += log(wt[j] - lo[j]); if (hu[j]) b_t += log(hi[j] - wt[j]); }
            const double ph_t = ft - mu * b_t;
            bool okk = (th_t == th_t) && (ph_t == ph_t) && fin(th_t) && fin(ph_t) && th_t <= theta_max;
            if (okk) for (int i = 0; i < nfilt; ++i) if (th_t >= filt[2 * i] && ph_t >= filt[2 * i + 1]) { okk = false; break; }
            if (okk) {
                const bool sw = gphid < 0.0 && theta <= theta_min && alpha * pow(-gphid, 2.3) > pow(theta, 1.1);
                const double eps = 10.0 * 2.220446049250313e-16 * fabs(phi);
                if (sw) { if (ph_t - phi - eps <= 1e-8 * alpha * gphid) { accepted = true; ftype = true; } }
                else if (th_t <= (1.0 - 1e-5) * theta || ph_t - eps <= phi - 1e-8 * theta) accepted = true;
            }
            if (accepted) break;
            alpha *= 0.5;
        }
        if (!accepted) {                // feasibility restoration, same rules as ocp_accept
            if (theta < 1e-6 || resto_calls >= 3) { status = theta > 1e-4 ? 2 : -2; break; }
            if (!MPCB_TGT_RESTO) { status = TGT_NEEDS_RESTO; break; }
            if (nfilt < MPCB_MAXFILT) { filt[2 * nfilt] = (1.0 - 1e-5) * theta; filt[2 * nfilt + 1] = phi - 1e-8 * theta; nfilt++; }
            resto = true; resto_calls += 1; theta_entry = theta;
            continue;
        }
        if (!ftype && nfilt < MPCB_MAXFILT) { filt[2 * nfilt] = (1.0 - 1e-5) * theta; filt[2 * nfilt + 1] = phi - 1e-8 * theta; nfilt++; }
        for (int j = 0; j < NVT; ++j) {
            w[j] = wt[j];
            if (hl[j]) { const double dn = w[j] - lo[j]; zL[j] = fmax(fmin(zL[j] + az * dzL[j], 1e10 * mu / dn), mu / (1e10 * dn)); }
            if (hu[j]) { const double dn = hi[j] - w[j]; zU[j] = fmax(fmin(zU[j] + az * dzU[j], 1e10 * mu / dn), mu / (1e10 * dn)); }
        }
        for (int i = 0; i < MCS; ++i) y[i] += alpha * rhs[NVT + i];
        it += 1;
        evaluate = true;
    }
#if MPCB_SENS_TGT
    if constexpr (CAPTURE)
        if (status != TGT_NEEDS_RESTO) tgt_capture(par, w, y, zL, zU, lo, hi, hl, hu, J, Hp, status, cap);
#else
    (void)cap;
#endif
    if (o.honor_original_bounds) {
        for (int j = 0; j < NWS; ++j) w[j] = fmin(fmax(w[j], S.lbx[j]), S.ubx[j]);
        double ct[MCS];
        tgt_eval(w, par, y, false, &f, ct, nullptr, nullptr, nullptr);
    }
    for (int j = 0; j < NWS; ++j) w_io[j] = w[j];
    *fout = f; *status_out = status; *iters_out = it;
}

// Regular variant first; an instance whose line search fails is handed back with status TGT_NEEDS_RESTO and its
// initial guess restored, and solved again (cold start: the same iterates up to that point) by the restoration variant -
// on the device by a second kernel (k_target_resto) that exits at once for every other instance, so that the common
// kernel does not carry the restoration code (it doubles the solver's instruction footprint).
MPCB_HD void tgt_solve_regular(const double* par, double* w, double* fout, int* status_out, int* iters_out, const TgtShared& S) {
#if MPCB_DENSE_SH
    tgt_solve_t<true>(par, w, fout, status_out, iters_out, S);        // large models: one variant (compile time, stack)
#else
    double w0[NWS];
    for (int i = 0; i < NWS; ++i) w0[i] = w[i];
    tgt_solve_t<false>(par, w, fout, status_out, iters_out, S);
    if (*status_out == TGT_NEEDS_RESTO)
        for (int i = 0; i < NWS; ++i) w[i] = w0[i];
#endif
}
MPCB_HD void tgt_solve_resto(const double* par, double* w, double* fout, int* status_out, int* iters_out, const TgtShared& S) {
    if (*status_out == TGT_NEEDS_RESTO) tgt_solve_t<true>(par, w, fout, status_out, iters_out, S);
}
// host callers (tests, CPU baseline): both in sequence
MPCB_HD void tgt_solve(const double* par, double* w, double* fout, int* status_out, int* iters_out, const TgtShared& S) {
    tgt_solve_regular(par, w, fout, status_out, iters_out, S);
    tgt_solve_resto(par, w, fout, status_out, iters_out, S);
}

#if MPCB_SENS_TGT
// The capture of one instance (mpcb_target_sens_factor): the solve of mpcb_target from the same guess wss0 (not modified),
// in the same two variants; *st is TGT_NEEDS_RESTO between them, then the capture's status.
MPCB_HD void tgt_sens_regular(const double* par, const double* wss0, double* cap, int* st, const TgtShared& S) {
    double w[NWS], f; int status, iters;
    for (int i = 0; i < NWS; ++i) w[i] = wss0[i];
    tgt_solve_t<false, true>(par, w, &f, &status, &iters, S, cap);
    if (status == TGT_NEEDS_RESTO) { *st = status; return; }
    for (int i = 0; i < NWS; ++i) cap[TgtSensLayout::w + i] = w[i];
    *st = (int)cap[TgtSensLayout::head];
}
MPCB_HD void tgt_sens_resto(const double* par, const double* wss0, double* cap, int* st, const TgtShared& S) {
    if (*st != TGT_NEEDS_RESTO) return;
    double w[NWS], f; int status, iters;
    for (int i = 0; i < NWS; ++i) w[i] = wss0[i];
    tgt_solve_t<true, true>(par, w, &f, &status, &iters, S, cap);
    for (int i = 0; i < NWS; ++i) cap[TgtSensLayout::w + i] = w[i];
    *st = (int)cap[TgtSensLayout::head];
}

// JVP: dw = -[K^{-1} dF/dtheta_ss dth]_{0:NWS};  VJP: K v = [gw; 0], g = -dF/dtheta_ss' v (K is symmetric)
MPCB_HD void tgt_jvp_dir(const double* cap, const double* th, double* dw) {
    if (cap[TgtSensLayout::head] != 0.0) { for (int i = 0; i < NWS; ++i) dw[i] = NAN; return; }
    const double* F = cap + TgtSensLayout::fth;
    double r[NKS]; int ipiv[NKS];
    for (int i = 0; i < NKS; ++i) {
        double a = 0.0;
        for (int t = 0; t < NTS; ++t) a -= F[i + NKS * t] * th[t];
        r[i] = a; ipiv[i] = (int)cap[TgtSensLayout::piv + i];
    }
    bk_solve<NKS>(cap + TgtSensLayout::K, ipiv, r);
    for (int i = 0; i < NWS; ++i) dw[i] = r[i];
}
MPCB_HD void tgt_vjp_inst(const double* cap, const double* gw, double* g) {
    if (cap[TgtSensLayout::head] != 0.0) { for (int t = 0; t < NTS; ++t) g[t] = NAN; return; }
    const double* F = cap + TgtSensLayout::fth;
    double r[NKS]; int ipiv[NKS];
    for (int i = 0; i < NKS; ++i) { r[i] = i < NWS ? gw[i] : 0.0; ipiv[i] = (int)cap[TgtSensLayout::piv + i]; }
    bk_solve<NKS>(cap + TgtSensLayout::K, ipiv, r);
    for (int t = 0; t < NTS; ++t) {
        double a = 0.0;
        for (int i = 0; i < NKS; ++i) a -= F[i + NKS * t] * r[i];
        g[t] = a;
    }
}
#endif  // MPCB_SENS_TGT
#endif  // MPCB_HAS_TARGET

// ---------------------------------------------------------------------------------------------
// Estimator update for one instance.  xi = [x; d] (nxi), P row-major nxi x nxi.
// ---------------------------------------------------------------------------------------------
struct EstShared { const double *Q, *R, *K, *dmin, *dmax; int has_dbounds; };

MPCB_HD void est_update(int est_type, const double* y_meas, const double* u, double t, const double* px,
                        const double* py, double* xi, double* P, const EstShared& E) {
    double x[NX], d[ND + 1], ul[NU], pxl[NPX + 1], pyl[NPY + 1];
    for (int i = 0; i < NX; ++i) x[i] = xi[i];
    for (int i = 0; i < ND; ++i) d[i] = (NXI > NX) ? xi[NX + i] : 0.0;
    for (int i = 0; i < NU; ++i) ul[i] = u[i];
    for (int i = 0; i < NPX; ++i) pxl[i] = px[i];
    for (int i = 0; i < NPY; ++i) pyl[i] = py[i];
    double yhat[NY], C[NY * NXI], e[NY];
    mdl_fy_xi(x, ul, d, &t, pyl, yhat, C);                        // C column-major NY x NXI
    for (int i = 0; i < NY; ++i) e[i] = y_meas[i] - yhat[i];
    if (est_type == 0) {                                          // Estimator.py:253-259
        for (int i = 0; i < NXI; ++i) {
            double a = xi[i];
            for (int j = 0; j < NY; ++j) a += E.K[i * NY + j] * e[j];
            xi[i] = a;
        }
    } else {                                                      // Estimator.py:288-309 / 340-381
        double PCt[NXI * NY], Sm[NY * NY], L[NY * NY];
        for (int i = 0; i < NXI; ++i)
            for (int j = 0; j < NY; ++j) {
                double a = 0.0;
                for (int l = 0; l < NXI; ++l) a += P[i * NXI + l] * C[j + NY * l];
                PCt[i * NY + j] = a;
            }
        for (int i = 0; i < NY; ++i)
            for (int j = 0; j < NY; ++j) {
                double a = E.R[i * NY + j];
                for (int l = 0; l < NXI; ++l) a += C[i + NY * l] * PCt[l * NY + j];
                Sm[i * NY + j] = a;
            }
        // K = P C' S^{-1}: general LU with partial pivoting on S' (K S = P C'  <=>  S' K' = (P C')'), as the
        // reference's `solve(S.T, (P C').T).T` (Estimator.py:297,352).  S is NOT symmetrised: the term C E C' of an
        // antisymmetric round-off E in P is what makes the error map E -> A(I-KC) E (I-KC)'A' contract; dropping it
        // lets E grow like |eig(A)|^2 per step for an open-loop unstable model.
        int piv[NY];
        for (int i = 0; i < NY; ++i)
            for (int j = 0; j < NY; ++j) L[i * NY + j] = Sm[j * NY + i];         // L := S'
        for (int c = 0; c < NY; ++c) {
            int pr = c; double best = fabs(L[c * NY + c]);
            for (int i = c + 1; i < NY; ++i) if (fabs(L[i * NY + c]) > best) { best = fabs(L[i * NY + c]); pr = i; }
            piv[c] = pr;
            if (pr != c) for (int j = 0; j < NY; ++j) { double tmp = L[c * NY + j]; L[c * NY + j] = L[pr * NY + j]; L[pr * NY + j] = tmp; }
            double inv = 1.0 / L[c * NY + c];
            for (int i = c + 1; i < NY; ++i) {
                double f = L[i * NY + c] * inv;
                L[i * NY + c] = f;
                for (int j = c + 1; j < NY; ++j) L[i * NY + j] -= f * L[c * NY + j];
            }
        }
        double Kg[NXI * NY];
        for (int r = 0; r < NXI; ++r) {
            double yv[NY];
            for (int i = 0; i < NY; ++i) yv[i] = PCt[r * NY + i];
            for (int c = 0; c < NY; ++c) if (piv[c] != c) { double tmp = yv[c]; yv[c] = yv[piv[c]]; yv[piv[c]] = tmp; }
            for (int i = 1; i < NY; ++i) {
                double a = yv[i];
                for (int l = 0; l < i; ++l) a -= L[i * NY + l] * yv[l];
                yv[i] = a;
            }
            for (int i = NY - 1; i >= 0; --i) {
                double a = yv[i];
                for (int l = i + 1; l < NY; ++l) a -= L[i * NY + l] * yv[l];
                yv[i] = a / L[i * NY + i];
            }
            for (int i = 0; i < NY; ++i) Kg[r * NY + i] = yv[i];
        }
        // P_corr = P - K (C P) ; xi += K e
        double CP[NY * NXI], Pc[NXI * NXI];
        for (int i = 0; i < NY; ++i)
            for (int j = 0; j < NXI; ++j) {
                double a = 0.0;
                for (int l = 0; l < NXI; ++l) a += C[i + NY * l] * P[l * NXI + j];
                CP[i * NXI + j] = a;
            }
        for (int i = 0; i < NXI; ++i) {
            double a = xi[i];
            for (int j = 0; j < NY; ++j) a += Kg[i * NY + j] * e[j];
            xi[i] = a;
            for (int j = 0; j < NXI; ++j) {
                double m = P[i * NXI + j];
                for (int l = 0; l < NY; ++l) m -= Kg[i * NY + l] * CP[l * NXI + j];
                Pc[i * NXI + j] = m;
            }
        }
        // A at the corrected state, previous input (Estimator.py:376); P+ = A Pc A' + Q
        for (int i = 0; i < NX; ++i) x[i] = xi[i];
        for (int i = 0; i < ND; ++i) d[i] = (NXI > NX) ? xi[NX + i] : 0.0;
        double Axi[NXI * NXI], AP[NXI * NXI];
        dyn_jac_xi(x, ul, d, pxl, t, Axi);
        for (int i = 0; i < NXI; ++i)
            for (int j = 0; j < NXI; ++j) {
                double a = 0.0;
                for (int l = 0; l < NXI; ++l) a += Axi[i * NXI + l] * Pc[l * NXI + j];
                AP[i * NXI + j] = a;
            }
        for (int i = 0; i < NXI; ++i)
            for (int j = 0; j < NXI; ++j) {
                double a = E.Q[i * NXI + j];
                for (int l = 0; l < NXI; ++l) a += AP[i * NXI + l] * Axi[j * NXI + l];
                P[i * NXI + j] = a;
            }
    }
    if (E.has_dbounds && NXI > NX)                                // MPC_code.py:659-665
        for (int i = 0; i < ND; ++i) xi[NX + i] = fmin(fmax(xi[NX + i], E.dmin[i]), E.dmax[i]);
}

// ---------------------------------------------------------------------------------------------
// Plant: measurement and one step (MPC_code.py:531-534, 813-816)
// ---------------------------------------------------------------------------------------------
#if !MPCB_PLANT_NOMINAL
MPCB_HD void plant_meas(const double* x, const double* u, double t, const double* pyp, const double* pymp, double* y) {
    double xl[MPCB_NXP], ul[NU], a[MPCB_NPYP + 1], b[MPCB_NPYP + 1];
    for (int i = 0; i < MPCB_NXP; ++i) xl[i] = x[i];
    for (int i = 0; i < NU; ++i) ul[i] = u[i];
    for (int i = 0; i < MPCB_NPYP; ++i) { a[i] = pyp[i]; b[i] = pymp[i]; }
    plt_fy(xl, ul, a, &t, b, y);
}
MPCB_HD void plant_step(double* x, const double* u, double t0, const double* pxp, const double* pxmp) {
    double xc[MPCB_NXP], ul[NU], a[MPCB_NPXP + 1], b[MPCB_NPXP + 1];
    for (int i = 0; i < MPCB_NXP; ++i) xc[i] = x[i];
    for (int i = 0; i < NU; ++i) ul[i] = u[i];
    for (int i = 0; i < MPCB_NPXP; ++i) { a[i] = pxp[i]; b[i] = pxmp[i]; }
#if MPCB_PLANT_RK4
    const double hs = MPCB_HSTEP / MPCB_PMX;
    for (int j = 0; j < MPCB_PMX; ++j) {
        double k1[MPCB_NXP], k2[MPCB_NXP], k3[MPCB_NXP], k4[MPCB_NXP], xt[MPCB_NXP];
        double t = t0 + j * hs, tt;
        plt_f(xc, ul, a, &t, b, k1);
        for (int i = 0; i < MPCB_NXP; ++i) xt[i] = xc[i] + 0.5 * hs * k1[i];
        tt = t + 0.5 * hs;
        plt_f(xt, ul, a, &tt, b, k2);
        for (int i = 0; i < MPCB_NXP; ++i) xt[i] = xc[i] + 0.5 * hs * k2[i];
        plt_f(xt, ul, a, &tt, b, k3);
        for (int i = 0; i < MPCB_NXP; ++i) xt[i] = xc[i] + hs * k3[i];
        tt = t + hs;
        plt_f(xt, ul, a, &tt, b, k4);
        for (int i = 0; i < MPCB_NXP; ++i) xc[i] += (hs / 6.0) * (k1[i] + 2.0 * k2[i] + 2.0 * k3[i] + k4[i]);
    }
    double post[MPCB_NXP];
    plt_post(a, b, post);
    for (int i = 0; i < MPCB_NXP; ++i) x[i] = xc[i] + post[i];
#else
    double xn[MPCB_NXP];
    plt_F(xc, ul, a, &t0, b, xn);
    for (int i = 0; i < MPCB_NXP; ++i) x[i] = xn[i];
#endif
}
#endif
