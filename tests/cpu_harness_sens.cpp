// cpu_harness_sens.cpp - TEST INFRASTRUCTURE: the OCP sensitivities of mpc-code_b200/csrc/mpcb_sens.cuh on the CPU
// (compiled with g++, no CUDA), after a solve with the same tick schedule as the kernel driver in mpcb_api.cu.  It lets
// the `-m "not gpu"` tests check the device arithmetic of the factor / JVP / VJP against the oracle without a GPU.
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
long h_sens_size(void) { return SensLayout::total; }

// Solve (bounds in the reference layout, IPOPT options as h_ocp of cpu_harness.cpp), then factor the sensitivities
// (fac_out: B x h_sens_size() doubles, may be null) and run the JVP of ndir directions dtheta [B, ndir, NTH] ->
// dw [B, ndir, NW] and the VJP gw [B, NW] -> gtheta [B, NTH].  sstatus: the factor's per-instance status.
int h_ocp_sens(int B, const double* par, double* w, double* f, int* status, int* iters,
               const double* lbx, const double* ubx, const double* lbg, const double* ubg,
               int max_iter, double tol, double mu_init, double relax, int honor,
               int ndir, const double* dtheta, double* dw, const double* gw, double* gtheta, int* sstatus, double* fac_out) {
    std::vector<double> lbi(NWI, -INFINITY), ubi(NWI, INFINITY);
    for (int k = 0; k <= NH; ++k) {
        for (int i = 0; i < NX; ++i) { lbi[k * NZA + i] = lbx[k * NZ + i]; ubi[k * NZA + i] = ubx[k * NZ + i]; }
        if (k < NH) for (int i = 0; i < NU; ++i) { lbi[k * NZA + NXA + i] = lbx[k * NZ + NX + i]; ubi[k * NZA + NXA + i] = ubx[k * NZ + NX + i]; }
    }
    OcpShared S; S.lbx = lbi.data(); S.ubx = ubi.data(); S.lbg = lbg; S.ubg = ubg;
    S.o.max_iter = max_iter; S.o.tol = tol; S.o.mu_init = mu_init; S.o.bound_relax = relax; S.o.bound_push = 1e-2;
    S.o.acceptable_tol = 1e-6; S.o.honor_original_bounds = honor; S.o.acceptable_iter = 15;
    std::vector<double> ws((size_t)B * OcpLayout::total, 0.0), fac((size_t)B * SensLayout::total, 0.0);
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
    for (int inst = 0; inst < B; ++inst) {
        OcpInst I = view(inst);
        for (int k = 0; k <= NH; ++k) ocp_export_stage(I, k);
        f[inst] = st[inst].fval; status[inst] = st[inst].status; iters[inst] = st[inst].iter;
        double scratch[KktScratch::total];
        double* fi = fac.data() + (size_t)inst * SensLayout::total;
        sstatus[inst] = ocp_sens_factor(I, fi, scratch);
        for (int r = 0; r < ndir; ++r)
            sens_jvp_dir(fi, dtheta + ((size_t)inst * ndir + r) * NTH, dw + ((size_t)inst * ndir + r) * NW);
        sens_vjp_inst(fi, gw + (size_t)inst * NW, gtheta + (size_t)inst * NTH);
    }
    if (fac_out) memcpy(fac_out, fac.data(), sizeof(double) * fac.size());
    return 0;
}
#endif

}  // extern "C"
