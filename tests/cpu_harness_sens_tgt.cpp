// cpu_harness_sens_tgt.cpp - TEST INFRASTRUCTURE: the sensitivities of the target problem of
// mpc-code_b200/csrc/mpcb_target.cuh (mpcb_target_sens_factor / mpcb_target_jvp / mpcb_target_vjp) on the CPU (compiled
// with g++, no CUDA).  It lets the `-m "not gpu"` tests of tests/test_target_sensitivity.py check the device arithmetic
// without a GPU.  It is NOT part of the product: nothing in mpc-code_b200/ loads it.
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "mpcb_target.cuh"

extern "C" {

long h_tgt_sens_size(void) {
#if MPCB_SENS_TGT
    return TgtSensLayout::total;
#else
    return -1;
#endif
}

long h_tgt_ntheta(void) {
#if MPCB_SENS_TGT
    return NTS;
#else
    return -1;
#endif
}

// Solve as mpcb_target (w0 -> w, status), then the capture as mpcb_target_sens_factor from the same w0 (sstatus,
// fac [B * h_tgt_sens_size()] when fac_out is given), the JVP of ndir directions dth [B, ndir, ntheta_ss] -> dw
// [B, ndir, nwss] and the VJP gw [B, nwss] -> gth [B, ntheta_ss].  Returns -1 without target sensitivities.
int h_target_sens(int B, const double* par, const double* w0, double* w, int* status, int* sstatus,
                  const double* lbx, const double* ubx, int max_iter, double tol, double mu_init, double relax, int honor,
                  int ndir, const double* dth, double* dw, const double* gw, double* gth, double* fac_out) {
#if MPCB_SENS_TGT
    TgtShared S; S.lbx = lbx; S.ubx = ubx;
    S.o.max_iter = max_iter; S.o.tol = tol; S.o.mu_init = mu_init; S.o.bound_relax = relax; S.o.bound_push = 1e-2;
    S.o.acceptable_tol = 1e-6; S.o.honor_original_bounds = honor; S.o.acceptable_iter = 15;
    std::vector<double> fac((size_t)B * TgtSensLayout::total, 0.0);
    for (int inst = 0; inst < B; ++inst) {
        const double* pi = par + (size_t)inst * MPCB_NPARSS;
        double* wi = w + (size_t)inst * NWS;
        double f; int iters;
        for (int i = 0; i < NWS; ++i) wi[i] = w0[(size_t)inst * NWS + i];
        tgt_solve(pi, wi, &f, status + inst, &iters, S);
        double* ci = fac.data() + (size_t)inst * TgtSensLayout::total;
        tgt_sens_regular(pi, w0 + (size_t)inst * NWS, ci, sstatus + inst, S);
        tgt_sens_resto(pi, w0 + (size_t)inst * NWS, ci, sstatus + inst, S);
        for (int r = 0; r < ndir; ++r)
            tgt_jvp_dir(ci, dth + ((size_t)inst * ndir + r) * NTS, dw + ((size_t)inst * ndir + r) * NWS);
        tgt_vjp_inst(ci, gw + (size_t)inst * NWS, gth + (size_t)inst * NTS);
    }
    if (fac_out) memcpy(fac_out, fac.data(), sizeof(double) * fac.size());
    return 0;
#else
    (void)B; (void)par; (void)w0; (void)w; (void)status; (void)sstatus; (void)lbx; (void)ubx; (void)max_iter; (void)tol;
    (void)mu_init; (void)relax; (void)honor; (void)ndir; (void)dth; (void)dw; (void)gw; (void)gth; (void)fac_out;
    return -1;
#endif
}

}  // extern "C"
