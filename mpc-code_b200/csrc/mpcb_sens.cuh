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
#if defined(__CUDA_ARCH__) && (MPCB_KKT_LANES > 1)
#  define S_LANE ((int)(threadIdx.x & (MPCB_KKT_LANES - 1)))
#  define S_NL   MPCB_KKT_LANES
#  define S_MASK (MPCB_KKT_LANES == 32 ? 0xffffffffu : \
                  (((1u << (MPCB_KKT_LANES & 31)) - 1u) << ((threadIdx.x & 31) & ~(MPCB_KKT_LANES - 1))))
#  define S_SYNC() __syncwarp(S_MASK)
#else
#  define S_LANE 0
#  define S_NL   1
#  define S_SYNC()
#endif

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
    const int lane = S_LANE;
    const int solve_status = I.st->status;
    if (solve_status != 0 && solve_status != 1) {
        if (lane == 0) fac[SensLayout::head] = 1.0;
        S_SYNC();
        return 1;
    }
    // mixed blocks (stage-parallel over the lanes) and the [A|B] blocks
    for (int k = lane; k <= NH; k += S_NL) {
        if (k == NH) { sens_mixed_term(I, fac + SensLayout::qt, fac + SensLayout::rt); continue; }
        sens_mixed_stage(I, k, fac + SensLayout::q + k * NZA * NTH);
        for (int e = 0; e < NXA * NZA; ++e) fac[SensLayout::ab + k * NXA * NZA + e] = I.rec[k * REC_SZ + R_AB + e];
    }
    S_SYNC();
    // backward Riccati sweep with delta_w = 0; its forward records (K, P_{k+1}, Gamma, Pi_{k+1}) go to fac
    OcpInst Ic = I;
    Ic.frec = fac + SensLayout::frec;
    KktIo io;
#if KKT_USE_TMA
    io.init(sm, lane);
    S_SYNC();
#endif
    bool ok = ocp_riccati(Ic, I.st->mu, 0.0, sm, io);
    S_SYNC();
    // Cholesky factors of R~_k = M_uu + B' P_{k+1} B (stage-parallel; the sweep keeps them only in registers)
    bool pd = ok;
    for (int k = lane; ok && k < NH; k += S_NL) {
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
#if defined(__CUDA_ARCH__) && (MPCB_KKT_LANES > 1)
    pd = __all_sync(S_MASK, pd) != 0;          // over the lanes of this instance only
#endif
#if MPCB_TERMCONS
    // Gramian of the terminal equality (no delta_c): Cholesky factor; Pi_0 (the sweep swaps its two Pi buffers per stage)
    if (ok) {
        const double* Gm = sm + KktScratch::Gm;
        const double* Pi = sm + ((NH % 2 == 0) ? KktScratch::PiA : KktScratch::PiB);
        double Gs[NXT * NXT], Lg[NXT * NXT], Lgi[NXT];
        for (int j = 0; j < NXT; ++j) for (int i = 0; i < NXT; ++i) Gs[i + NXT * j] = 0.5 * (Gm[i + NXT * j] + Gm[j + NXT * i]);
        if (!sens_chol<NXT>(Gs, Lg, Lgi)) pd = false;
        S_SYNC();
        if (lane == 0) {
            for (int e = 0; e < NXT * NXT; ++e) fac[SensLayout::gl + e] = Lg[e];
            for (int e = 0; e < NXA * NXT; ++e) fac[SensLayout::pi0 + e] = Pi[e];
        }
    }
#endif
    const int status = (ok && pd) ? 0 : 2;
    S_SYNC();
    if (lane == 0) fac[SensLayout::head] = (double)status;
    S_SYNC();
    return status;
}

// ---- sweeps ---------------------------------------------------------------------------------------------------------
// Solves the condensed KKT system for one right-hand side given by `src`:
//   src.q(k, q)   stage gradient (NZA),  src.pN(p)  terminal gradient (NXA),  src.rT(r)  terminal-equality residual,
//   src.z0(z)     fixed dz_0,            src.y(k, dz, du) / src.yN(dz)  receive the solution,  src.p0(p0)  costate of z_0
// Everything is read from fac; kk holds the feed-forward terms between the two sweeps.
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
        for (int j = 0; j < NZA; ++j) { double a = q[j]; for (int l = 0; l < NXA; ++l) a += AB[l + NXA * j] * p[l]; q[j] = a; }
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
