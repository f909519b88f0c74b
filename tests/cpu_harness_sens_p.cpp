// cpu_harness_sens_p.cpp - TEST INFRASTRUCTURE: the OCP sensitivities with respect to p = [d | px | py] of
// mpc-code_b200/csrc/mpcb_sens.cuh (mpcb_ocp_sens_factor_p / mpcb_ocp_jvp_p / mpcb_ocp_vjp_p) on the CPU (compiled with
// g++, no CUDA), after a solve with the same tick schedule as the kernel driver in mpcb_api.cu.  It lets the `-m "not gpu"`
// tests of tests/test_ocp_sensitivity_params.py check the device arithmetic without a GPU.
// It is NOT part of the product: nothing in mpc-code_b200/ loads it.
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "mpcb_target.cuh"
#if MPCB_HAS_OCP
#include "mpcb_sens.cuh"
#endif

extern "C" {

#if MPCB_HAS_OCP
long h_sens_size_theta(void) { return SensLayout::total; }

long h_sens_size_p(void) {
#if MPCB_SENS_P
    return SensLayout::total + SensPLayout::total;
#else
    return -1;
#endif
}

// As h_ocp_sens of cpu_harness_sens.cpp, for p = [d | px | py] (include/mpcb.h, mpcb_ocp_sens_factor_p): the capture fac [B * h_sens_size_p()]
// is the B theta captures followed by the B p-blocks.  theta_only = 1 writes only the theta part into a zero-filled
// capture, as mpcb_ocp_sens_factor would.  Also runs the theta JVP / VJP on the same capture (dtheta / gtheta).
// Returns -1 when the problem has no p-blocks (MPCB_SENS_P = 0).
int h_ocp_sens_p(int B, const double* par, double* w, double* f, int* status, int* iters,
                 const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                 int max_iter, double tol, double mu_init, double relax, int honor, int theta_only,
                 int ndir, const double* dp, double* dw, const double* gw, double* gp,
                 int ndir_th, const double* dtheta, double* dw_th, double* gtheta, int* sstatus, double* fac_out) {
#if MPCB_SENS_P
    std::vector<double> lbi(NWI, -INFINITY), ubi(NWI, INFINITY);
    for (int k = 0; k <= NH; ++k) {
        for (int i = 0; i < NX; ++i) { lbi[k * NZA + i] = lbx[k * NZ + i]; ubi[k * NZA + i] = ubx[k * NZ + i]; }
        if (k < NH) for (int i = 0; i < NU; ++i) { lbi[k * NZA + NXA + i] = lbx[k * NZ + NX + i]; ubi[k * NZA + NXA + i] = ubx[k * NZ + NX + i]; }
    }
    OcpShared S; S.lbx = lbi.data(); S.ubx = ubi.data(); S.lbg = lbg; S.ubg = ubg;
    S.o.max_iter = max_iter; S.o.tol = tol; S.o.mu_init = mu_init; S.o.bound_relax = relax; S.o.bound_push = 1e-2;
    S.o.acceptable_tol = 1e-6; S.o.honor_original_bounds = honor; S.o.acceptable_iter = 15;
    std::vector<double> ws((size_t)B * OcpLayout::total, 0.0), fac((size_t)B * (SensLayout::total + SensPLayout::total), 0.0);
    std::vector<InstState> st(B);
    auto view = [&](int inst) { return ocp_inst(ws.data() + (size_t)inst * OcpLayout::total, w + (size_t)inst * NW,
                                                par + (size_t)inst * NPAR, &st[inst]); };
    for (int inst = 0; inst < B; ++inst) for (int k = 0; k <= NH; ++k) { OcpInst I = view(inst); ocp_init_stage(I, S, k); }
    for (int ticks = 0; ticks < (max_iter + 2) * 8; ++ticks) {
        int active = 0;
        for (int inst = 0; inst < B; ++inst) {
            OcpInst I = view(inst);
            double scratch[KktScratch::total];
            if (st[inst].state == ST_EVAL) { for (int k = 0; k < NH; ++k) ocp_eval_stage(I, S, k); ocp_kkt(I, S, scratch); }
            if (st[inst].state == ST_LS) { for (int k = 0; k < NH; ++k) ocp_trial_stage(I, S, k); ocp_accept(I, S); }
            if (st[inst].state != ST_DONE) active++;
        }
        if (!active) break;
    }
    double* pblk = fac.data() + (size_t)B * SensLayout::total;
    for (int inst = 0; inst < B; ++inst) {
        OcpInst I = view(inst);
        for (int k = 0; k <= NH; ++k) ocp_export_stage(I, k);
        f[inst] = st[inst].fval; status[inst] = st[inst].status; iters[inst] = st[inst].iter;
        double scratch[KktScratch::total];
        double* fi = fac.data() + (size_t)inst * SensLayout::total;
        sstatus[inst] = ocp_sens_factor(I, fi, scratch);
        if (!theta_only)
            for (int k = 0; k <= NH; ++k) ocp_sens_pblocks(I, k, fi, pblk + (size_t)inst * SensPLayout::total);
    }
    for (int inst = 0; inst < B; ++inst) {
        const double* fi = fac.data() + (size_t)inst * SensLayout::total;
        const double* pi = pblk + (size_t)inst * SensPLayout::total;
        for (int r = 0; r < ndir; ++r)
            sens_jvp_p_dir(fi, pi, dp + ((size_t)inst * ndir + r) * NPP, dw + ((size_t)inst * ndir + r) * NW);
        sens_vjp_p_inst(fi, pi, gw + (size_t)inst * NW, gp + (size_t)inst * NPP);
        for (int r = 0; r < ndir_th; ++r)
            sens_jvp_dir(fi, dtheta + ((size_t)inst * ndir_th + r) * NTH, dw_th + ((size_t)inst * ndir_th + r) * NW);
        sens_vjp_inst(fi, gw + (size_t)inst * NW, gtheta + (size_t)inst * NTH);
    }
    if (fac_out) memcpy(fac_out, fac.data(), sizeof(double) * fac.size());
    return 0;
#else
    (void)B; (void)par; (void)w; (void)f; (void)status; (void)iters; (void)lbx; (void)ubx; (void)lbg; (void)ubg;
    (void)max_iter; (void)tol; (void)mu_init; (void)relax; (void)honor; (void)theta_only; (void)ndir; (void)dp; (void)dw;
    (void)gw; (void)gp; (void)ndir_th; (void)dtheta; (void)dw_th; (void)gtheta; (void)sstatus; (void)fac_out;
    return -1;
#endif
}
#endif

}  // extern "C"
