// mpcb_sens.cuh - parametric sensitivity of the batched OCP solution (sIPOPT-style), after a solve.
//
// theta = [x_hat (NX) | x_s (NX) | u_s (NU) | u_{k-1} (NU)] = par[0 : 2NX+NU] and par[OFF_UM1 : OFF_UM1+NU].
// At the returned iterate the primal-dual barrier system F(v; theta) = 0 is differentiated: dv/dtheta =
// -(dF/dv)^{-1} dF/dtheta, with the bound multipliers and range-row slacks condensed exactly as in the Newton step
// (Sigma = Z / D, no regularisation) and x_0 eliminated (dz_0 = [dx_hat; du_{k-1}]).  The condensed KKT matrix is the
// one whose blocks the solve's last evaluation left in the stage records, so its factorisation is one Riccati sweep
// with delta_w = 0 (ocp_riccati, unchanged).  theta does not enter the dynamics, so every right-hand side has zero
// defects: a JVP / VJP is one backward vector sweep, the terminal-equality multiplier solve and one forward sweep.
//
//   ocp_sens_factor   per instance (lanes as ocp_kkt): mixed blocks d(grad L)/dtheta at w*, Riccati factors -> fac
//   sens_jvp_dir      per (instance, direction): dw = J dtheta in the caller's layout
//   sens_vjp_inst     per instance: gtheta = J' gw
// The capture buffer `fac` holds everything the sweeps read, so they stay valid after the handle has solved again.
#pragma once
#include "mpcb_ocp.cuh"

#define NTH MPCB_NTH                      // 2 (NX + NU)
#ifdef __CUDACC__
#  define SENS_M __host__ __device__ __forceinline__       // (non-static) member functions
#else
#  define SENS_M inline
#endif
#ifndef MPCB_SENS_CONT_DEP
#define MPCB_SENS_CONT_DEP 0              // 1: the ContForm integrand depends on theta (no generated mixed derivatives)
#endif

// Capture layout (doubles per instance), in the order the sweeps read it.  The per-stage Riccati quantities are written
// by ocp_riccati itself, as its forward records (K_k, P_{k+1}, Gamma_k, Pi_{k+1} at FREC_* of stage k).
struct SensLayout {
    static constexpr int head = 0;                                   // [0] status (0 / 1 / 2 as a double)
    static constexpr int frec = 2;                                   // NH * FREC_SZ
    static constexpr int ab = frec + NH * FREC_SZ;                   // NH * NXA*NZA  [A_k | B_k]
    static constexpr int chol = ab + NH * NXA * NZA;                 // NH * (NU*NU + NU)  Cholesky factor of R~_k, 1/diag
    static constexpr int q = chol + NH * (NU * NU + NU);             // NH * NZA*NTH  d(grad_z L_k)/dtheta + G'Sigma_s dg/dtheta
    static constexpr int qt = q + NH * NZA * NTH;                    // NXA*NTH  d(grad V_f)/dtheta
    static constexpr int rt = qt + NXA * NTH;                        // NXT*NTH  d(terminal equality)/dtheta
    static constexpr int gl = rt + NXT * NTH;                        // NXT*NXT  Cholesky factor of the TermCons Gramian
    static constexpr int pi0 = gl + NXT * NXT;                       // NXA*NXT  Pi_0
    static constexpr int total = (pi0 + NXA * NXT + 1) / 2 * 2;
};

// theta component -> parameter index, and the fixed initial stage state z_0 = [x_hat; u_{k-1}] of a direction
MPCB_HD int sens_par_index(int t) { return t < 2 * NX + NU ? t : MPCB_OFF_UM1 + (t - (2 * NX + NU)); }
MPCB_HD double sens_z0(const double* th, int i) { return i < NX ? th[i] : th[2 * NX + NU + (i - NX)]; }

// ---- mixed blocks at w* ------------------------------------------------------------------------------------------
// stage k: Q = d(grad_{z,u} l_k)/dtheta + d(mult' grad R_k)/dtheta + G_k' Sigma_s dR_k/dtheta   (NZA x NTH, column-major)
MPCB_HD void sens_mixed_stage(const OcpInst& I, int k, double* Q) {
    double z[NXA], u[NU], d[ND + 1], px[NPX + 1], py[NPY + 1], t0;
    for (int i = 0; i < NXA; ++i) z[i] = I.w[k * NZA + i];
    for (int i = 0; i < NU; ++i) u[i] = I.w[k * NZA + NXA + i];
    stage_params(I.par, k, d, px, py, &t0);
    ocp_cost_dth(z, u, I.par, px, py, Q);
#if NG > 0
    double Yt[NG * NTH], HYt[NZA * NTH];
    ocp_out_dth(z, u, I.par, px, py, I.ym + k * NG, Yt, HYt);
    const double* R = I.rec + k * REC_SZ;
    for (int t = 0; t < NTH; ++t)
        for (int j = 0; j < NZA; ++j) {
            double a = HYt[j + NZA * t];
            for (int r = 0; r < NG; ++r) a += R[R_G + r + NG * j] * R[R_SG + r] * Yt[r + NG * t];
            Q[j + NZA * t] += a;
        }
#endif
}

// terminal: d(grad V_f)/dtheta (NXA x NTH; the carried inputs of z_N do not enter V_f) and d(r_T)/dtheta (NXT x NTH)
MPCB_HD void sens_mixed_term(const OcpInst& I, double* QT, double* RT) {
    double Tt[NX * NTH];
    ocp_term_dth(I.w + NH * NZA, I.par, Tt);
    for (int t = 0; t < NTH; ++t)
        for (int i = 0; i < NXA; ++i) QT[i + NXA * t] = i < NX ? Tt[i + NX * t] : 0.0;
#if MPCB_TERMCONS
    ocp_termc_dth(I.w + NH * NZA, I.par, RT);
#else
    (void)RT;
#endif
}

// ---- factor: one instance, lanes as in ocp_kkt (ocp_riccati runs on them) ----------------------------------------
// Cholesky L L' = A of an n x n SPD matrix (column-major, lower part read); Li = 1 / diag(L).  False if not SPD.
template <int n>
MPCB_HD bool sens_chol(const double* A, double* L, double* Li) {
    for (int j = 0; j < n; ++j) {
        double djj = A[j + n * j];
        for (int l = 0; l < j; ++l) djj -= L[j + n * l] * L[j + n * l];
        if (!(djj > 0.0)) return false;
        const double s = sqrt(djj);
        L[j + n * j] = s; Li[j] = 1.0 / s;
        for (int i = j + 1; i < n; ++i) {
            double a = A[i + n * j];
            for (int l = 0; l < j; ++l) a -= L[i + n * l] * L[j + n * l];
            L[i + n * j] = a * Li[j];
        }
        for (int i = 0; i < j; ++i) L[i + n * j] = 0.0;
    }
    return true;
}
template <int n>
MPCB_HD void sens_chol_solve(const double* L, const double* Li, double* b) {     // b <- (L L')^{-1} b
    for (int i = 0; i < n; ++i) { double a = b[i]; for (int l = 0; l < i; ++l) a -= L[i + n * l] * b[l]; b[i] = a * Li[i]; }
    for (int i = n - 1; i >= 0; --i) { double a = b[i]; for (int l = i + 1; l < n; ++l) a -= L[l + n * i] * b[l]; b[i] = a * Li[i]; }
}

// Status: 0 computed, 1 the solve did not end with status 0 / 1, 2 wrong inertia at delta_w = 0.
MPCB_HD int ocp_sens_factor(const OcpInst& I, double* fac, double* sm) {
    const int lane = KktLanes::id();
    const int solve_status = I.st->status;
    if (solve_status != 0 && solve_status != 1) {
        if (lane == 0) fac[SensLayout::head] = 1.0;
        KktLanes::sync();
        return 1;
    }
    // mixed blocks (stage-parallel over the lanes) and the [A|B] blocks
    for (int k = lane; k <= NH; k += KktLanes::n) {
        if (k == NH) { sens_mixed_term(I, fac + SensLayout::qt, fac + SensLayout::rt); continue; }
        sens_mixed_stage(I, k, fac + SensLayout::q + k * NZA * NTH);
        for (int e = 0; e < NXA * NZA; ++e) fac[SensLayout::ab + k * NXA * NZA + e] = I.rec[k * REC_SZ + R_AB + e];
    }
    KktLanes::sync();
    // backward Riccati sweep with delta_w = 0; its forward records (K, P_{k+1}, Gamma, Pi_{k+1}) go to fac
    OcpInst Ic = I;
    Ic.frec = fac + SensLayout::frec;
    KktIo io;
#if KKT_USE_TMA
    io.init(sm, lane);
    KktLanes::sync();
#endif
    bool ok = ocp_riccati(Ic, I.st->mu, 0.0, sm, io);
    KktLanes::sync();
    // Cholesky factors of R~_k = M_uu + B' P_{k+1} B (stage-parallel; the sweep keeps them only in registers)
    bool pd = ok;
    for (int k = lane; ok && k < NH; k += KktLanes::n) {
        const double* R = I.rec + k * REC_SZ; const double* F = fac + SensLayout::frec + k * FREC_SZ;
        double Muu[NU * NU];
        for (int j = 0; j < NU; ++j)
            for (int i = 0; i < NU; ++i) {
                double a = R[R_M + (NXA + i) + NZA * (NXA + j)];
                for (int l = 0; l < NXA; ++l) {
                    double pb = 0.0;
                    for (int m = 0; m < NXA; ++m) pb += F[FREC_P + l + NXA * m] * R[R_AB + NXA * NXA + m + NXA * j];
                    a += R[R_AB + NXA * NXA + l + NXA * i] * pb;
                }
                Muu[i + NU * j] = a;
            }
        double* C = fac + SensLayout::chol + k * (NU * NU + NU);
        if (!sens_chol<NU>(Muu, C, C + NU * NU)) pd = false;
    }
    pd = KktLanes::all(pd);                    // over the lanes of this instance only
#if MPCB_TERMCONS
    // Gramian of the terminal equality (no delta_c): Cholesky factor; Pi_0 (the sweep swaps its two Pi buffers per stage)
    if (ok) {
        const double* Gm = sm + KktScratch::Gm;
        const double* Pi = sm + ((NH % 2 == 0) ? KktScratch::PiA : KktScratch::PiB);
        double Gs[NXT * NXT], Lg[NXT * NXT], Lgi[NXT];
        for (int j = 0; j < NXT; ++j) for (int i = 0; i < NXT; ++i) Gs[i + NXT * j] = 0.5 * (Gm[i + NXT * j] + Gm[j + NXT * i]);
        if (!sens_chol<NXT>(Gs, Lg, Lgi)) pd = false;
        KktLanes::sync();
        if (lane == 0) {
            for (int e = 0; e < NXT * NXT; ++e) fac[SensLayout::gl + e] = Lg[e];
            for (int e = 0; e < NXA * NXT; ++e) fac[SensLayout::pi0 + e] = Pi[e];
        }
    }
#endif
    const int status = (ok && pd) ? 0 : 2;
    KktLanes::sync();
    if (lane == 0) fac[SensLayout::head] = (double)status;
    KktLanes::sync();
    return status;
}

// ---- sweeps ---------------------------------------------------------------------------------------------------------
// Solves the condensed KKT system for one right-hand side given by `src`:
//   src.q(k, q)   stage gradient (NZA),  src.pN(p)  terminal gradient (NXA),  src.rT(r)  terminal-equality residual,
//   src.z0(z)     fixed dz_0,            src.y(k, dz, du) / src.yN(dz)  receive the solution,  src.p0(p0)  costate of z_0
// Sources with SensDefects<Src>::value (the p sweeps) also give the defect of the dynamics row of stage k and see the
// multiplier of that row:
//   src.c(k, c)   defect c_k (NXA):  dz_{k+1} = A_k dz_k + B_k du_k + c_k,
//   src.keep(k, p)  the backward costate p_k (k = 1..NH),  src.lam(k, dz_{k+1}, nu)  after dz_{k+1} is known.
// For the other sources the defect terms are not compiled: the theta sweeps keep their arithmetic.
// Everything is read from fac; kk holds the feed-forward terms between the two sweeps.
template <class Src> struct SensDefects { static constexpr bool value = false; };

template <class Src>
MPCB_HD void sens_sweep(const double* fac, Src& src, double* kk) {
    double p[NXA], q[NZA], nu[NXT + 1];
    src.pN(p);
#if MPCB_TERMCONS
    double h[NXT];
    for (int j = 0; j < NXT; ++j) h[j] = 0.0;
#endif
    for (int k = NH - 1; k >= 0; --k) {
        const double* AB = fac + SensLayout::ab + k * NXA * NZA;
        const double* F = fac + SensLayout::frec + k * FREC_SZ;
        const double* C = fac + SensLayout::chol + k * (NU * NU + NU);
        src.q(k, q);
        if constexpr (SensDefects<Src>::value) {
            // V_{k+1}(A dz + B du + c) contributes [A|B]'(P_{k+1} c + p_{k+1}); c reaches dz_N like B kf does
            double c[NXA], pc[NXA];
            src.keep(k + 1, p);
            src.c(k, c);
            for (int i = 0; i < NXA; ++i) { double a = p[i]; for (int m = 0; m < NXA; ++m) a += F[FREC_P + i + NXA * m] * c[m]; pc[i] = a; }
            for (int j = 0; j < NZA; ++j) { double a = q[j]; for (int l = 0; l < NXA; ++l) a += AB[l + NXA * j] * pc[l]; q[j] = a; }
#if MPCB_TERMCONS
            for (int j = 0; j < NXT; ++j) { double a = h[j]; for (int l = 0; l < NXA; ++l) a += F[FREC_PI + l + NXA * j] * c[l]; h[j] = a; }
#endif
        } else {
            for (int j = 0; j < NZA; ++j) { double a = q[j]; for (int l = 0; l < NXA; ++l) a += AB[l + NXA * j] * p[l]; q[j] = a; }
        }
        double* kf = kk + k * NU;
        for (int i = 0; i < NU; ++i) kf[i] = q[NXA + i];
        sens_chol_solve<NU>(C, C + NU * NU, kf);
        for (int i = 0; i < NU; ++i) kf[i] = -kf[i];
#if MPCB_TERMCONS
        for (int j = 0; j < NXT; ++j) {
            double a = h[j];
            for (int l = 0; l < NXA; ++l) {
                double bk = 0.0;
                for (int m = 0; m < NU; ++m) bk += AB[NXA * NXA + l + NXA * m] * kf[m];
                a += F[FREC_PI + l + NXA * j] * bk;
            }
            h[j] = a;
        }
#endif
        for (int i = 0; i < NXA; ++i) {
            double a = q[i];
            for (int m = 0; m < NU; ++m) a += F[FREC_K + m + NU * i] * q[NXA + m];
            p[i] = a;
        }
    }
    double dz[NXA], dn[NXA], du[NU];
    src.z0(dz);
#if MPCB_TERMCONS
    {   // G nu = h + Pi_0' dz_0 + r_T
        const double* Pi0 = fac + SensLayout::pi0; const double* Lg = fac + SensLayout::gl;
        double r[NXT], Lgi[NXT];
        src.rT(r);
        for (int j = 0; j < NXT; ++j) {
            double a = h[j] + r[j];
            for (int l = 0; l < NXA; ++l) a += Pi0[l + NXA * j] * dz[l];
            nu[j] = a; Lgi[j] = 1.0 / Lg[j + NXT * j];
        }
        sens_chol_solve<NXT>(Lg, Lgi, nu);
        for (int i = 0; i < NXA; ++i) { double a = p[i]; for (int j = 0; j < NXT; ++j) a += Pi0[i + NXA * j] * nu[j]; p[i] = a; }
    }
#endif
    src.p0(p);
    for (int k = 0; k < NH; ++k) {
        const double* AB = fac + SensLayout::ab + k * NXA * NZA;
        const double* F = fac + SensLayout::frec + k * FREC_SZ;
        for (int i = 0; i < NU; ++i) {
            double a = kk[k * NU + i];
            for (int j = 0; j < NXA; ++j) a += F[FREC_K + i + NU * j] * dz[j];
#if MPCB_TERMCONS
            for (int j = 0; j < NXT; ++j) a += F[FREC_GA + i + NU * j] * nu[j];
#endif
            du[i] = a;
        }
        src.y(k, dz, du);
        for (int i = 0; i < NXA; ++i) {
            double a = 0.0;
            for (int j = 0; j < NXA; ++j) a += AB[i + NXA * j] * dz[j];
            for (int j = 0; j < NU; ++j) a += AB[NXA * NXA + i + NXA * j] * du[j];
            dn[i] = a;
        }
        if constexpr (SensDefects<Src>::value) {
            double c[NXA];
            src.c(k, c);
            for (int i = 0; i < NXA; ++i) dn[i] += c[i];
            src.lam(k, dn, nu);
        }
        for (int i = 0; i < NXA; ++i) dz[i] = dn[i];
    }
    src.yN(dz, nu);
}

// JVP: q_k = Q_k dtheta, p_N = Q_T dtheta, r_T = R_T dtheta, dz_0 from dtheta; writes dw (caller's layout, NW)
struct SensJvpSrc {
    const double* fac; const double* th; double* dw;
    SENS_M void q(int k, double* q) const {
        const double* Q = fac + SensLayout::q + k * NZA * NTH;
        for (int j = 0; j < NZA; ++j) { double a = 0.0; for (int t = 0; t < NTH; ++t) a += Q[j + NZA * t] * th[t]; q[j] = a; }
    }
    SENS_M void pN(double* p) const {
        const double* Q = fac + SensLayout::qt;
        for (int j = 0; j < NXA; ++j) { double a = 0.0; for (int t = 0; t < NTH; ++t) a += Q[j + NXA * t] * th[t]; p[j] = a; }
    }
    SENS_M void rT(double* r) const {
        const double* Q = fac + SensLayout::rt;
        for (int j = 0; j < NXT; ++j) { double a = 0.0; for (int t = 0; t < NTH; ++t) a += Q[j + NXT * t] * th[t]; r[j] = a; }
    }
    SENS_M void z0(double* z) const { for (int i = 0; i < NXA; ++i) z[i] = sens_z0(th, i); }
    SENS_M void p0(const double*) const {}
    SENS_M void y(int k, const double* dz, const double* du) const {
        for (int i = 0; i < NX; ++i) dw[k * NZ + i] = dz[i];
        for (int i = 0; i < NU; ++i) dw[k * NZ + NX + i] = du[i];
    }
    SENS_M void yN(const double* dz, const double*) const { for (int i = 0; i < NX; ++i) dw[NH * NZ + i] = dz[i]; }
};

// VJP: the same system with the gradient -gw (dz_0 = 0, r_T = 0); then gtheta = -sum_k Q_k' y_k - Q_T' y_N - R_T' nu
// plus, on the z_0 components, the multiplier of z_0 = dz_0:  -(p_0 + Pi_0 nu)  (it contains the direct gw[z_0] term).
struct SensVjpSrc {
    const double* fac; const double* gw; double* g;
    SENS_M void q(int k, double* q) const {
        for (int i = 0; i < NXA; ++i) q[i] = i < NX ? -gw[k * NZ + i] : 0.0;
        for (int i = 0; i < NU; ++i) q[NXA + i] = -gw[k * NZ + NX + i];
    }
    SENS_M void pN(double* p) const { for (int i = 0; i < NXA; ++i) p[i] = i < NX ? -gw[NH * NZ + i] : 0.0; }
    SENS_M void rT(double* r) const { for (int j = 0; j < NXT; ++j) r[j] = 0.0; }
    SENS_M void z0(double* z) const { for (int i = 0; i < NXA; ++i) z[i] = 0.0; }
    SENS_M void p0(const double* p) const {
        for (int t = 0; t < NTH; ++t) g[t] = 0.0;
        for (int i = 0; i < NX; ++i) g[i] = -p[i];
        for (int i = NX; i < NXA; ++i) g[2 * NX + NU + (i - NX)] = -p[i];
    }
    SENS_M void y(int k, const double* dz, const double* du) const {
        const double* Q = fac + SensLayout::q + k * NZA * NTH;
        for (int t = 0; t < NTH; ++t) {
            double a = 0.0;
            for (int j = 0; j < NXA; ++j) a += Q[j + NZA * t] * dz[j];
            for (int j = 0; j < NU; ++j) a += Q[NXA + j + NZA * t] * du[j];
            g[t] -= a;
        }
    }
    SENS_M void yN(const double* dz, const double* nu) const {
        const double* Q = fac + SensLayout::qt; const double* R = fac + SensLayout::rt;
        for (int t = 0; t < NTH; ++t) {
            double a = 0.0;
            for (int j = 0; j < NXA; ++j) a += Q[j + NXA * t] * dz[j];
            for (int j = 0; j < NXT; ++j) a += R[j + NXT * t] * nu[j];
            g[t] -= a;
        }
    }
};

MPCB_HD void sens_jvp_dir(const double* fac, const double* th, double* dw) {
    if (fac[SensLayout::head] != 0.0) { for (int i = 0; i < NW; ++i) dw[i] = NAN; return; }
    double kk[NH * NU];
    SensJvpSrc s{fac, th, dw};
    sens_sweep(fac, s, kk);
}

MPCB_HD void sens_vjp_inst(const double* fac, const double* gw, double* gth) {
    if (fac[SensLayout::head] != 0.0) { for (int t = 0; t < NTH; ++t) gth[t] = NAN; return; }
    double kk[NH * NU];
    SensVjpSrc s{fac, gw, gth};
    sens_sweep(fac, s, kk);
}

// =====================================================================================================================
// Sensitivities with respect to the parameters that enter the dynamics:
//   p = [d (ND) | px_0 .. px_{NH-1} (NPX NH) | py_0 .. py_{NH-1} (NPY NH)] = par[OFF_D : OFF_D+ND] ++ par[OFF_PX : NPAR].
// Stage k depends on p_k = [d; px_k; py_k] only (NPK columns), the terminal maps on d.  p enters the dynamics rows, so
// the right-hand sides have defects c_k = Fp_k dp_k.  The capture of mpcb_ocp_sens_factor_p is the theta capture of
// all B instances, unchanged, followed by the p-blocks of all B instances (SensPLayout each); fac[1] of an instance's
// theta capture is 1 when its p-blocks were written.
//   ocp_sens_pblocks  per (instance, stage k = 0..NH), the mapping of ocp_eval_stage: Fp_k, Qp_k, terminal d-blocks
//   sens_jvp_p_dir    per (instance, direction): dw = J_p dp
//   sens_vjp_p_inst   per instance: gp = J_p' gw
// =====================================================================================================================
#ifndef MPCB_SENS_P
#define MPCB_SENS_P 0                     // 0: the problem cannot provide the p-blocks (decided by the generator)
#endif
#define NPK (ND + NPX + NPY)              // columns of p_k = [d; px_k; py_k]
#define NPM (ND + NPX)                    // the model's parameters [d; px]: the first NPM columns of p_k
#define NPP (ND + (NPX + NPY) * NH)       // n_p

struct SensPLayout {                                                 // doubles per instance, after the B theta captures
    static constexpr int fp = 0;                                     // NH * NXA*NPK  dF_k/dp_k (rows of v_k = u_{k-1}: 0)
    static constexpr int qp = fp + NH * NXA * NPK;                   // NH * NZA*NPK  d(grad L_k)/dp_k + G'Sigma_s dR_k/dp_k
    static constexpr int qt = qp + NH * NZA * NPK;                   // NXA*ND  d(grad V_f)/dd
    static constexpr int rt = qt + NXA * ND;                         // NXT*ND  d(terminal equality)/dd
    static constexpr int total = (rt + NXT * ND + 1) / 2 * 2;
};

// local column c of p_k -> index into p
MPCB_HD int sens_p_index(int k, int c) {
    return c < ND ? c : (c < NPM ? ND + k * NPX + (c - ND) : ND + NPX * NH + k * NPY + (c - NPM));
}

// sens_dyn_dp also gives the d / px columns of the target problem's model equalities (mpcb_target.cuh, MPCB_SENS_TGT)
#if MPCB_SENS_P || MPCB_SENS_TGT
#if MPCB_DYN_RK4 && MPCB_SENS_NQ > 0
// The model ODE on the augmented state [x; q], q' = 0: q holds the components MPCB_SENS_QIDX of [d; px] that the
// right-hand side reads (the generated mdlp_* take them from the state, the rest from the context).  Run with the
// adjoint seed [lam; 0], the RK4 sweeps of the solve give dx_N/dq in the q columns of S and the mixed Hessian of lam' x_N.
#ifndef MPCB_MDLP_NC
#define MPCB_MDLP_NC 0
#endif
#ifndef MPCB_MDLP_NR
#define MPCB_MDLP_NR 0
#endif
struct SysModelP {
    static constexpr int NS = NX + MPCB_SENS_NQ, NM = MX, NC = MPCB_MDLP_NC, NR = MPCB_MDLP_NR;
    typedef ModelCtx Ctx;
#if MPCB_MDLP_NC + MPCB_MDLP_NR > 0
    MPCB_HDM void f_c(const double* x, const Ctx& c, double t, double* o, double* cache) { mdlp_f_c(x, c.u, c.d, &t, c.px, o, cache); }
    MPCB_HDM void f_rc(const double* x, const Ctx& c, double t, const double* cache, double* o, double* rc) {
        mdlp_f_rc(x, c.u, c.d, &t, c.px, cache, o, rc);
    }
    MPCB_HDM void f_rcp(const double* x, const Ctx& c, double t, const double* cache, double* rc) { mdlp_f_rcp(x, c.u, c.d, &t, c.px, cache, rc); }
    MPCB_HDM void f_vjp_c(const double* x, const Ctx& c, double t, const double* nu, const double* cache, const double* rc, double* o) {
        mdlp_f_vjp_c(x, c.u, c.d, &t, c.px, nu, cache, rc, o);
    }
    MPCB_HDM void f_sh_c(const double* x, const Ctx& c, double t, const double* S, const double* nu, const double* cache,
                         const double* rc, double* o, double* K, double* Hc) {
        mdlp_f_sh_c(x, c.u, c.d, &t, c.px, S, nu, cache, rc, o, K, Hc);
    }
#endif
    MPCB_HDM void f(const double* x, const Ctx& c, double t, double* o) { mdlp_f(x, c.u, c.d, &t, c.px, o); }
    MPCB_HDM void f_vjp(const double* x, const Ctx& c, double t, const double* nu, double* o) { mdlp_f_vjp(x, c.u, c.d, &t, c.px, nu, o); }
    MPCB_HDM void f_sh(const double* x, const Ctx& c, double t, const double* S, const double* nu, double* o, double* K, double* Hc) {
        mdlp_f_sh(x, c.u, c.d, &t, c.px, S, nu, o, K, Hc);
    }
};
#endif

// Fm = dx_{k+1}/d[d; px] (NX x NPM) and Hm = d(grad_{x,u} lam' x_{k+1})/d[d; px] (NZ x NPM), column-major
MPCB_HD void sens_dyn_dp(const double* x, const double* u, const double* d, const double* px, double t0, const double* lam,
                         double* Fm, double* Hm) {
#if MPCB_DYN_RK4
    for (int e = 0; e < NX * NPM; ++e) Fm[e] = 0.0;
    for (int e = 0; e < NZ * NPM; ++e) Hm[e] = 0.0;
#if MPCB_SENS_NQ > 0
    {
        constexpr int NQ = MPCB_SENS_NQ, NS = NX + NQ, NZS = NS + NU;
        constexpr int qi[NQ] = MPCB_SENS_QIDX;
        ModelCtx c; c.u = u; c.d = d; c.px = px;
        double xt[NS], lt[NS], xe[NS], S[NS * NZS], Ht[NZS * (NZS + 1) / 2], lbuf[RkSize<SysModelP>::TOTAL];
        for (int i = 0; i < NX; ++i) { xt[i] = x[i]; lt[i] = lam[i]; }
        for (int j = 0; j < NQ; ++j) { xt[NX + j] = qi[j] < ND ? d[qi[j]] : px[qi[j] - ND]; lt[NX + j] = 0.0; }
        for (int e = 0; e < NZS * (NZS + 1) / 2; ++e) Ht[e] = 0.0;
        rk4_full_t<SysModelP>(xt, c, t0, lt, xe, S, Ht, RkBuf{lbuf, 1});
        for (int j = 0; j < NQ; ++j) {
            for (int i = 0; i < NX; ++i) Fm[i + NX * qi[j]] = S[i + NS * (NX + j)];
            for (int r = 0; r < NZ; ++r) Hm[r + NZ * qi[j]] = Ht[tri(r < NX ? r : r + NQ, NX + j)];
        }
    }
#endif
    double Jp[NX * NPM + 1];
    mdl_post_dp(d, px, Jp);
    for (int e = 0; e < NX * NPM; ++e) Fm[e] += Jp[e];
#else
    mdl_F_dp(x, u, d, &t0, px, lam, Fm, Hm);
#endif
}
#endif  // MPCB_SENS_P || MPCB_SENS_TGT

#if MPCB_SENS_P

// stage k: Fp (NXA x NPK) and Qp (NZA x NPK) at w*, with the multipliers the stage record was built with
MPCB_HD void sens_p_stage(const OcpInst& I, int k, double* Fp, double* Qp) {
    double z[NXA], u[NU], lam[NXA], d[ND + 1], px[NPX + 1], py[NPY + 1], t0;
    for (int i = 0; i < NXA; ++i) { z[i] = I.w[k * NZA + i]; lam[i] = I.lam[k * NXA + i]; }
    for (int i = 0; i < NU; ++i) u[i] = I.w[k * NZA + NXA + i];
    stage_params(I.par, k, d, px, py, &t0);
    ocp_cost_dp(z, u, I.par, px, py, Qp);
#if NG > 0
    {
        double Yp[NG * NPK], HYp[NZA * NPK];
        ocp_out_dp(z, u, I.par, px, py, I.ym + k * NG, Yp, HYp);
        const double* R = I.rec + k * REC_SZ;
        for (int c = 0; c < NPK; ++c)
            for (int j = 0; j < NZA; ++j) {
                double a = HYp[j + NZA * c];
                for (int r = 0; r < NG; ++r) a += R[R_G + r + NG * j] * R[R_SG + r] * Yp[r + NG * c];
                Qp[j + NZA * c] += a;
            }
    }
#endif
    double Fm[NX * NPM + 1], Hm[NZ * NPM + 1];
    sens_dyn_dp(z, u, d, px, t0, lam, Fm, Hm);
    for (int e = 0; e < NXA * NPK; ++e) Fp[e] = 0.0;
    for (int c = 0; c < NPM; ++c) {
        for (int i = 0; i < NX; ++i) Fp[i + NXA * c] = Fm[i + NX * c];
        for (int r = 0; r < NZ; ++r) Qp[(r < NX ? r : r + NAUG) + NZA * c] += Hm[r + NZ * c];     // model (x, u) -> (x, v, u)
    }
}

// terminal: d(grad V_f)/dd (NXA x ND) and d(r_T)/dd (NXT x ND)
MPCB_HD void sens_p_term(const OcpInst& I, double* QT, double* RT) {
    double Tp[NX * ND + 1];
    ocp_term_dp(I.w + NH * NZA, I.par, Tp);
    for (int c = 0; c < ND; ++c)
        for (int i = 0; i < NXA; ++i) QT[i + NXA * c] = i < NX ? Tp[i + NX * c] : 0.0;
#if MPCB_TERMCONS
    ocp_termc_dp(I.w + NH * NZA, I.par, RT);
#else
    (void)RT;
#endif
}

// one (instance, k) of the p-blocks: fac = the instance's theta capture, pb = its p-blocks
MPCB_HD void ocp_sens_pblocks(const OcpInst& I, int k, double* fac, double* pb) {
    const int solve_status = I.st->status;
    if (solve_status == 0 || solve_status == 1) {
        if (k < NH) sens_p_stage(I, k, pb + SensPLayout::fp + k * NXA * NPK, pb + SensPLayout::qp + k * NZA * NPK);
        else sens_p_term(I, pb + SensPLayout::qt, pb + SensPLayout::rt);
    }
    if (k == 0) fac[1] = 1.0;
}

// JVP: q_k = Qp_k dp_k, c_k = Fp_k dp_k, p_N = QT dd, r_T = RT dd, dz_0 = 0; writes dw (caller's layout, NW)
struct SensJvpPSrc {
    const double* pb; const double* dp; double* dw;
    SENS_M void loc(int k, double* v) const { for (int c = 0; c < NPK; ++c) v[c] = dp[sens_p_index(k, c)]; }
    SENS_M void q(int k, double* q) const {
        const double* Q = pb + SensPLayout::qp + k * NZA * NPK;
        double v[NPK];
        loc(k, v);
        for (int j = 0; j < NZA; ++j) { double a = 0.0; for (int c = 0; c < NPK; ++c) a += Q[j + NZA * c] * v[c]; q[j] = a; }
    }
    SENS_M void c(int k, double* cv) const {
        const double* Fp = pb + SensPLayout::fp + k * NXA * NPK;
        double v[NPK];
        loc(k, v);
        for (int i = 0; i < NXA; ++i) { double a = 0.0; for (int c = 0; c < NPK; ++c) a += Fp[i + NXA * c] * v[c]; cv[i] = a; }
    }
    SENS_M void pN(double* p) const {
        const double* Q = pb + SensPLayout::qt;
        for (int j = 0; j < NXA; ++j) { double a = 0.0; for (int c = 0; c < ND; ++c) a += Q[j + NXA * c] * dp[c]; p[j] = a; }
    }
    SENS_M void rT(double* r) const {
        const double* Q = pb + SensPLayout::rt;
        for (int j = 0; j < NXT; ++j) { double a = 0.0; for (int c = 0; c < ND; ++c) a += Q[j + NXT * c] * dp[c]; r[j] = a; }
    }
    SENS_M void z0(double* z) const { for (int i = 0; i < NXA; ++i) z[i] = 0.0; }
    SENS_M void p0(const double*) const {}
    SENS_M void keep(int, const double*) const {}
    SENS_M void lam(int, const double*, const double*) const {}
    SENS_M void y(int k, const double* dz, const double* du) const {
        for (int i = 0; i < NX; ++i) dw[k * NZ + i] = dz[i];
        for (int i = 0; i < NU; ++i) dw[k * NZ + NX + i] = du[i];
    }
    SENS_M void yN(const double* dz, const double*) const { for (int i = 0; i < NX; ++i) dw[NH * NZ + i] = dz[i]; }
};

// VJP: the system with the gradient -gw and no defects; with its solution (y, lam^, nu)
//   gp = -sum_k (Qp_k' y_k + Fp_k' lam^_k) - QT' y_N - RT' nu,   lam^_k = P_{k+1} dz_{k+1} + p_{k+1} + Pi_{k+1} nu,
// the multiplier of the dynamics row of stage k (p_{k+1} of the backward sweep is kept per stage).
struct SensVjpPSrc {
    const double* fac; const double* pb; const double* gw; double* g; double* pk;      // pk: (NH + 1) * NXA
    SENS_M void q(int k, double* q) const {
        for (int i = 0; i < NXA; ++i) q[i] = i < NX ? -gw[k * NZ + i] : 0.0;
        for (int i = 0; i < NU; ++i) q[NXA + i] = -gw[k * NZ + NX + i];
    }
    SENS_M void c(int, double* cv) const { for (int i = 0; i < NXA; ++i) cv[i] = 0.0; }
    SENS_M void pN(double* p) const { for (int i = 0; i < NXA; ++i) p[i] = i < NX ? -gw[NH * NZ + i] : 0.0; }
    SENS_M void rT(double* r) const { for (int j = 0; j < NXT; ++j) r[j] = 0.0; }
    SENS_M void z0(double* z) const { for (int i = 0; i < NXA; ++i) z[i] = 0.0; }
    SENS_M void p0(const double*) const {}
    SENS_M void keep(int k, const double* p) const { for (int i = 0; i < NXA; ++i) pk[k * NXA + i] = p[i]; }
    SENS_M void y(int k, const double* dz, const double* du) const {
        const double* Q = pb + SensPLayout::qp + k * NZA * NPK;
        for (int c = 0; c < NPK; ++c) {
            double a = 0.0;
            for (int j = 0; j < NXA; ++j) a += Q[j + NZA * c] * dz[j];
            for (int j = 0; j < NU; ++j) a += Q[NXA + j + NZA * c] * du[j];
            g[sens_p_index(k, c)] -= a;
        }
    }
    SENS_M void lam(int k, const double* dn, const double* nu) const {
        const double* F = fac + SensLayout::frec + k * FREC_SZ;
        const double* Fp = pb + SensPLayout::fp + k * NXA * NPK;
        double l[NXA];
        for (int i = 0; i < NXA; ++i) {
            double a = pk[(k + 1) * NXA + i];
            for (int m = 0; m < NXA; ++m) a += F[FREC_P + i + NXA * m] * dn[m];
#if MPCB_TERMCONS
            for (int j = 0; j < NXT; ++j) a += F[FREC_PI + i + NXA * j] * nu[j];
#else
            (void)nu;
#endif
            l[i] = a;
        }
        for (int c = 0; c < NPK; ++c) {
            double a = 0.0;
            for (int i = 0; i < NXA; ++i) a += Fp[i + NXA * c] * l[i];
            g[sens_p_index(k, c)] -= a;
        }
    }
    SENS_M void yN(const double* dz, const double* nu) const {
        const double* Q = pb + SensPLayout::qt; const double* R = pb + SensPLayout::rt;
        for (int c = 0; c < ND; ++c) {
            double a = 0.0;
            for (int j = 0; j < NXA; ++j) a += Q[j + NXA * c] * dz[j];
            for (int j = 0; j < NXT; ++j) a += R[j + NXT * c] * nu[j];
            g[c] -= a;
        }
    }
};
template <> struct SensDefects<SensJvpPSrc> { static constexpr bool value = true; };
template <> struct SensDefects<SensVjpPSrc> { static constexpr bool value = true; };

MPCB_HD bool sens_p_valid(const double* fac) { return fac[SensLayout::head] == 0.0 && fac[1] == 1.0; }

MPCB_HD void sens_jvp_p_dir(const double* fac, const double* pb, const double* dp, double* dw) {
    if (!sens_p_valid(fac)) { for (int i = 0; i < NW; ++i) dw[i] = NAN; return; }
    double kk[NH * NU];
    SensJvpPSrc s{pb, dp, dw};
    sens_sweep(fac, s, kk);
}

MPCB_HD void sens_vjp_p_inst(const double* fac, const double* pb, const double* gw, double* gp) {
    if (!sens_p_valid(fac)) { for (int t = 0; t < NPP; ++t) gp[t] = NAN; return; }
    for (int t = 0; t < NPP; ++t) gp[t] = 0.0;
    double kk[NH * NU], pk[(NH + 1) * NXA];
    SensVjpPSrc s{fac, pb, gw, gp, pk};
    sens_sweep(fac, s, kk);
}
#endif  // MPCB_SENS_P
