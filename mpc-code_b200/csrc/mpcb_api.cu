// mpcb_api.cu - kernels and the C ABI of include/mpcb.h for ONE compiled problem.
//
// Built per problem as  nvcc -gencode arch=compute_100a,code=sm_100a -I<dir with mpcb_model.h> ...
// The generated mpcb_model.h carries the sizes and the user's model as __device__ functions.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <string>
#include <utility>
#include <vector>
#include "mpcb.h"
#include "mpcb_target.cuh"
#if MPCB_HAS_OCP
#include "mpcb_sens.cuh"
#endif

#define MPCB_NKERNELS 8
enum { KC_OCP_INIT = 0, KC_OCP_EVAL = 1, KC_OCP_KKT = 2, KC_OCP_TRIAL = 3, KC_OCP_ACCEPT = 4, KC_TARGET = 5, KC_ESTIMATE = 6, KC_OTHER = 7 };

// launch shape of the stage-parallel kernels (tunable at build time: tools/tune_eval.py)
#ifndef MPCB_EVAL_BLOCK
#define MPCB_EVAL_BLOCK 128
#endif
#ifndef MPCB_EVAL_MINBLOCKS
// 2 blocks of 128 threads per SM: 254 registers per thread, no spills.  Measured on B200 (Ex_NMPC, profiles/r02_variants_*.txt):
// 3 blocks (168 registers, the sweeps' matrices spilling) 32.4 ms of evaluation per 10 steps, 2 blocks 25.0, 9 blocks of 32
// threads at 224 registers 25.2, 11 at 184 registers 29.5 - occupancy beyond 8 warps does not pay for the spills.
#define MPCB_EVAL_MINBLOCKS 2
#endif

#ifndef MPCB_FLOPS_TABLE
#define MPCB_FLOPS_TABLE
#endif

// ---------------------------------------------------------------------------------------------
// kernels (thin wrappers; the arithmetic lives in the host/device functions of the .cuh files)
// ---------------------------------------------------------------------------------------------
#if MPCB_HAS_OCP
struct OcpArgs {
    int B;
    const double* par; double* w; double* ws; InstState* st;
    unsigned long long* counters;      // [0] instance-evaluations (derivatives), [1] instance-trials (line search)
    OcpShared S;
};

__device__ __forceinline__ OcpInst ocp_view(const OcpArgs& a, int inst) {
    return ocp_inst(a.ws + (size_t)inst * OcpLayout::total, a.w + (size_t)inst * NW, a.par + (size_t)inst * NPAR, a.st + inst);
}

__global__ void __launch_bounds__(128) k_ocp_init(OcpArgs a) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = tid / (NH + 1), k = tid % (NH + 1);
    if (inst >= a.B) return;
    OcpInst I = ocp_view(a, inst);
    ocp_init_stage(I, a.S, k);
}

// The sub-step records of the RK4 sweeps (EVAL_RK_DOUBLES per thread) live in shared memory when MINBLOCKS blocks of
// them fit one SM (227 kB; Ex_NMPC: 70 doubles x 128 threads x 2 blocks = 140 kB), otherwise in thread-local memory.
#ifndef MPCB_EVAL_SMEM
#define MPCB_EVAL_SMEM ((EVAL_RK_DOUBLES) > 0 && \
                        ((size_t)(EVAL_RK_DOUBLES) * 8 * MPCB_EVAL_BLOCK + 1024) * MPCB_EVAL_MINBLOCKS <= 232448)
#endif
#define EVAL_SMEM_BYTES (MPCB_EVAL_SMEM ? (size_t)(EVAL_RK_DOUBLES) * 8 * MPCB_EVAL_BLOCK : 0)
#ifdef MPCB_EVAL_MAXNREG
#define EVAL_BOUNDS __maxnreg__(MPCB_EVAL_MAXNREG)
#else
#define EVAL_BOUNDS __launch_bounds__(MPCB_EVAL_BLOCK, MPCB_EVAL_MINBLOCKS)
#endif
__global__ void EVAL_BOUNDS k_ocp_eval(OcpArgs a) {
    extern __shared__ double eval_smem[];
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = tid / NH, k = tid % NH;
    if (inst >= a.B) return;
    if (a.st[inst].state != ST_EVAL) return;
    if (k == 0) atomicAdd(a.counters, 1ULL);
    OcpInst I = ocp_view(a, inst);
    ocp_eval_stage<MPCB_EVAL_SMEM>(I, a.S, k, RkBuf{eval_smem + threadIdx.x, MPCB_EVAL_BLOCK});
}

#if MPCB_EVAL_FIRST
// first tick of a solve: all multipliers are zero (see ocp_eval_stage<., FIRST>)
__global__ void __launch_bounds__(128) k_ocp_eval_first(OcpArgs a) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = tid / NH, k = tid % NH;
    if (inst >= a.B) return;
    if (a.st[inst].state != ST_EVAL) return;
    if (k == 0) atomicAdd(a.counters, 1ULL);
    OcpInst I = ocp_view(a, inst);
    ocp_eval_stage<false, true>(I, a.S, k);
}
#endif

#ifndef MPCB_TGT_BLOCK
#define MPCB_TGT_BLOCK 64       // threads per block of the one-thread-per-instance target solve
#endif
#ifndef KKT_WARPS
// warps per block of the KKT kernel: as many as fit the 48 kB of static shared memory, at most 4
#define KKT_SCRATCH_BYTES ((int)sizeof(double) * KktScratch::total * (32 / MPCB_KKT_LANES))
#define KKT_WARPS (4 * KKT_SCRATCH_BYTES <= 48 * 1024 ? 4 : (2 * KKT_SCRATCH_BYTES <= 48 * 1024 ? 2 : 1))
#endif
// Per-instance kernels of the KKT mapping (k_ocp_kkt, k_ocp_sens_factor): KktLanes::n lanes per instance.  Lane groups
// run KKT_WARPS warps per block and keep their KktScratch in static shared memory, one row per group; one thread per
// instance runs blocks of 32 threads and keeps it thread-local.  KKT_SCRATCH(sm) declares `double* sm`.
#if MPCB_KKT_LANES > 1
#define KKT_THREADS (32 * KKT_WARPS)
static_assert(sizeof(double) * KktScratch::total * (KKT_THREADS / MPCB_KKT_LANES) <= 48 * 1024,
              "MPCB_KKT_LANES: the KKT scratch of the lane groups of one warp exceeds the 48 kB of static shared memory; "
              "this problem needs more lanes per instance or the one-thread mapping -DMPCB_KKT_LANES=1");
#define KKT_SCRATCH(sm) __shared__ __align__(16) double sm##_rows[KKT_THREADS / KktLanes::n][KktScratch::total]; \
                        double* sm = sm##_rows[threadIdx.x / KktLanes::n]
#else
#define KKT_THREADS 32
#define KKT_SCRATCH(sm) double sm[KktScratch::total]
#endif
#ifdef MPCB_KKT_MINBLOCKS
#define KKT_BOUNDS __launch_bounds__(KKT_THREADS, MPCB_KKT_MINBLOCKS)
#else
#define KKT_BOUNDS __launch_bounds__(KKT_THREADS)
#endif
#define KKT_GRID(B) nblk((long)(B) * MPCB_KKT_LANES, KKT_THREADS), KKT_THREADS

__global__ void KKT_BOUNDS k_ocp_kkt(OcpArgs a) {
    const int inst = (blockIdx.x * blockDim.x + threadIdx.x) / KktLanes::n;
    if (inst >= a.B) return;
    if (a.st[inst].state != ST_EVAL) return;
    KKT_SCRATCH(sm);
    OcpInst I = ocp_view(a, inst);
    ocp_kkt(I, a.S, sm);
}

__global__ void __launch_bounds__(128) k_ocp_trial(OcpArgs a) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = tid / NH, k = tid % NH;
    if (inst >= a.B) return;
    if (a.st[inst].state != ST_LS) return;
    if (k == 0) atomicAdd(a.counters + 1, 1ULL);
    OcpInst I = ocp_view(a, inst);
    ocp_trial_stage(I, a.S, k);
}

// n_active != null: count the instances that are not done after this tick
__global__ void __launch_bounds__(32 * KKT_WARPS) k_ocp_accept(OcpArgs a, int* n_active) {
    const int inst = (blockIdx.x * blockDim.x + threadIdx.x) / WarpLanes::n;
    if (inst >= a.B) return;
    if (a.st[inst].state == ST_LS) {
        OcpInst I = ocp_view(a, inst);
        ocp_accept(I, a.S);
    }
    if (n_active && threadIdx.x % WarpLanes::n == 0 && a.st[inst].state != ST_DONE) atomicAdd(n_active, 1);
}

// Loop condition of the device-driven solve (body of the CUDA-graph WHILE node, after k_ocp_accept): another tick while
// some instance still iterates.  ctr = {instances not done (reset here), ticks of this solve, ticks since creation}.
// `ticks` = number of ticks run since the previous call of this kernel.
__global__ void k_ocp_cond(cudaGraphConditionalHandle handle, int* n_active, unsigned long long* ctr, int max_ticks, int ticks) {
    const int active = *n_active;
    *n_active = 0;
    const unsigned long long t = (ctr[0] += (unsigned long long)ticks);
    ctr[1] += (unsigned long long)ticks;
    cudaGraphSetConditional(handle, (active > 0 && t < (unsigned long long)max_ticks) ? 1u : 0u);
}

__global__ void k_ocp_output(OcpArgs a, double* f, int* status, int* iters) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = tid / (NH + 1), k = tid % (NH + 1);
    if (inst >= a.B) return;
    OcpInst I = ocp_view(a, inst);
    ocp_export_stage(I, k);                 // internal iterate -> caller's w (reference layout)
    if (k == 0) { f[inst] = a.st[inst].fval; status[inst] = a.st[inst].status; iters[inst] = a.st[inst].iter; }
}

// stage derivatives alone (mpcb_stage_derivs)
__global__ void EVAL_BOUNDS k_stage_derivs(int B, const double* par, const double* w, const double* lam,
                                                      double* A, double* Bm, double* c, double* H) {
    extern __shared__ double eval_smem[];
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = tid / NH, k = tid % NH;
    if (inst >= B) return;
    const double* wi = w + (size_t)inst * NW; const double* pi = par + (size_t)inst * NPAR;
    double x[NX], u[NU], l[NX], d[ND + 1], px[NPX + 1], py[NPY + 1], t0;
    for (int i = 0; i < NX; ++i) { x[i] = wi[k * NZ + i]; l[i] = lam[((size_t)inst * NH + k) * NX + i]; }
    for (int i = 0; i < NU; ++i) u[i] = wi[k * NZ + NX + i];
    stage_params(pi, k, d, px, py, &t0);
    double xn[NX], Al[NX * NX], Bl[NX * NU], Hp[NZP];
    for (int i = 0; i < NZP; ++i) Hp[i] = 0.0;
    dyn_full<(MPCB_EVAL_SMEM && MPCB_DYN_RK4 && !MPCB_CONTFORM)>(x, u, d, px, t0, l, xn, Al, Bl, Hp, RkBuf{eval_smem + threadIdx.x, MPCB_EVAL_BLOCK});
    const size_t s = (size_t)inst * NH + k;
    for (int i = 0; i < NX * NX; ++i) A[s * NX * NX + i] = Al[i];
    for (int i = 0; i < NX * NU; ++i) Bm[s * NX * NU + i] = Bl[i];
    for (int i = 0; i < NX; ++i) c[s * NX + i] = xn[i] - wi[(k + 1) * NZ + i];
    for (int i = 0; i < NZP; ++i) H[s * NZP + i] = Hp[i];
}

// ---- sensitivities of the last OCP solve (mpcb_ocp_sens_factor / mpcb_ocp_jvp / mpcb_ocp_vjp) ----------------------
// factor: the mapping of k_ocp_kkt (ocp_riccati runs on the same lanes and the same shared-memory scratch)
__device__ __forceinline__ void sens_factor_inst(const double* ws, const double* par, InstState* st, double* fac, int* status,
                                                 int inst, double* sm) {
    OcpInst I = ocp_inst(const_cast<double*>(ws) + (size_t)inst * OcpLayout::total, nullptr, par + (size_t)inst * NPAR, st + inst);
    const int r = ocp_sens_factor(I, fac + (size_t)inst * SensLayout::total, sm);
    if (KktLanes::id() == 0) status[inst] = r;
}
__global__ void KKT_BOUNDS k_ocp_sens_factor(int B, const double* ws, const double* par, InstState* st, double* fac, int* status) {
    const int inst = (blockIdx.x * blockDim.x + threadIdx.x) / KktLanes::n;
    if (inst >= B) return;
    KKT_SCRATCH(sm);
    sens_factor_inst(ws, par, st, fac, status, inst, sm);
}
// JVP: one thread per (instance, direction); the directions of an instance sit on consecutive lanes, so their reads of
// the instance's capture are broadcasts.  VJP: one thread per instance.
__global__ void __launch_bounds__(128) k_ocp_jvp(int B, int ndir, const double* fac, const double* dth, double* dw) {
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= (long)B * ndir) return;
    const long inst = tid / ndir;
    sens_jvp_dir(fac + inst * SensLayout::total, dth + tid * NTH, dw + tid * NW);
}
__global__ void __launch_bounds__(128) k_ocp_vjp(int B, const double* fac, const double* gw, double* gth) {
    const long inst = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    sens_vjp_inst(fac + inst * SensLayout::total, gw + inst * NW, gth + inst * NTH);
}
#if MPCB_SENS_P
// p-blocks: one thread per (instance, stage k = 0..NH), the mapping of k_ocp_eval (k = NH: the terminal blocks).  The
// generated derivative code runs on independent threads, not on the lanes of a per-instance warp.
__global__ void __launch_bounds__(128) k_ocp_sens_pblocks(int B, const double* ws, const double* par, InstState* st, double* fac) {
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= (long)B * (NH + 1)) return;
    const long inst = tid / (NH + 1);
    const int k = (int)(tid % (NH + 1));
    OcpInst I = ocp_inst(const_cast<double*>(ws) + inst * OcpLayout::total, nullptr, par + inst * NPAR, st + inst);
    ocp_sens_pblocks(I, k, fac + inst * SensLayout::total, fac + (long)B * SensLayout::total + inst * SensPLayout::total);
}
__global__ void __launch_bounds__(128) k_ocp_jvp_p(int B, int ndir, const double* fac, const double* dp, double* dw) {
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= (long)B * ndir) return;
    const long inst = tid / ndir;
    sens_jvp_p_dir(fac + inst * SensLayout::total, fac + (long)B * SensLayout::total + inst * SensPLayout::total,
                   dp + tid * NPP, dw + tid * NW);
}
__global__ void __launch_bounds__(128) k_ocp_vjp_p(int B, const double* fac, const double* gw, double* gp) {
    const long inst = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    sens_vjp_p_inst(fac + inst * SensLayout::total, fac + (long)B * SensLayout::total + inst * SensPLayout::total,
                    gw + inst * NW, gp + inst * NPP);
}
#endif
#endif

#if MPCB_HAS_TARGET
__global__ void __launch_bounds__(64) k_target(int B, const double* par, double* w, double* f, int* status, int* iters,
                                               TgtShared S) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    tgt_solve_regular(par + (size_t)inst * MPCB_NPARSS, w + (size_t)inst * NWS, f + inst, status + inst, iters + inst, S);
}
// the rare instances whose line search failed: restoration variant (see tgt_solve_regular)
__global__ void __launch_bounds__(64) k_target_resto(int B, const double* par, double* w, double* f, int* status, int* iters,
                                                     TgtShared S) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    tgt_solve_resto(par + (size_t)inst * MPCB_NPARSS, w + (size_t)inst * NWS, f + inst, status + inst, iters + inst, S);
}
#if MPCB_SENS_TGT
// sensitivities of the target solution (mpcb_target_sens_factor): the mapping and the two variants of k_target
__global__ void __launch_bounds__(64) k_target_sens(int B, const double* par, const double* w0, double* fac, int* status,
                                                    TgtShared S) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    tgt_sens_regular(par + (size_t)inst * MPCB_NPARSS, w0 + (size_t)inst * NWS, fac + (size_t)inst * TgtSensLayout::total,
                     status + inst, S);
}
__global__ void __launch_bounds__(64) k_target_sens_resto(int B, const double* par, const double* w0, double* fac, int* status,
                                                          TgtShared S) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    tgt_sens_resto(par + (size_t)inst * MPCB_NPARSS, w0 + (size_t)inst * NWS, fac + (size_t)inst * TgtSensLayout::total,
                   status + inst, S);
}
// JVP: one thread per (instance, direction), as k_ocp_jvp; VJP: one thread per instance
__global__ void __launch_bounds__(128) k_target_jvp(int B, int ndir, const double* fac, const double* dth, double* dw) {
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= (long)B * ndir) return;
    const long inst = tid / ndir;
    tgt_jvp_dir(fac + inst * TgtSensLayout::total, dth + tid * NTS, dw + tid * NWS);
}
__global__ void __launch_bounds__(128) k_target_vjp(int B, const double* fac, const double* gw, double* gth) {
    const long inst = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    tgt_vjp_inst(fac + inst * TgtSensLayout::total, gw + inst * NWS, gth + inst * NTS);
}
#endif
#endif

__global__ void __launch_bounds__(64) k_estimate(int B, int est_type, const double* y, const double* u, const double* t,
                                                 const double* px, const double* py, double* xi, double* P, EstShared E) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    est_update(est_type, y + (size_t)inst * NY, u + (size_t)inst * NU, t[inst], px + (size_t)inst * NPX,
               py + (size_t)inst * NPY, xi + (size_t)inst * NXI, P + (size_t)inst * NXI * NXI, E);
}

__global__ void k_model_output(int B, const double* x, const double* u, const double* d, const double* t,
                               const double* py, double* y) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    double xl[NX], ul[NU], dl[ND + 1], pl[NPY + 1], yl[NY], tt = t[inst];
    for (int i = 0; i < NX; ++i) xl[i] = x[(size_t)inst * NX + i];
    for (int i = 0; i < NU; ++i) ul[i] = u[(size_t)inst * NU + i];
    for (int i = 0; i < ND; ++i) dl[i] = d[(size_t)inst * ND + i];
    for (int i = 0; i < NPY; ++i) pl[i] = py[(size_t)inst * NPY + i];
    mdl_fy(xl, ul, dl, &tt, pl, yl);
    for (int i = 0; i < NY; ++i) y[(size_t)inst * NY + i] = yl[i];
}

__global__ void k_model_step(int B, const double* x, const double* u, const double* d, const double* t,
                             const double* px, double* xn) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    double xl[NX], ul[NU], dl[ND + 1], pl[NPX + 1], xo[NX];
    for (int i = 0; i < NX; ++i) xl[i] = x[(size_t)inst * NX + i];
    for (int i = 0; i < NU; ++i) ul[i] = u[(size_t)inst * NU + i];
    for (int i = 0; i < ND; ++i) dl[i] = d[(size_t)inst * ND + i];
    for (int i = 0; i < NPX; ++i) pl[i] = px[(size_t)inst * NPX + i];
    dyn_value(xl, ul, dl, pl, t[inst], xo);
    for (int i = 0; i < NX; ++i) xn[(size_t)inst * NX + i] = xo[i];
}

#if !MPCB_PLANT_NOMINAL
__global__ void k_plant_meas(int B, const double* x, const double* u, const double* t, const double* pyp,
                             const double* pymp, const double* noise, double* y) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    double yl[NY];
    plant_meas(x + (size_t)inst * MPCB_NXP, u + (size_t)inst * NU, t[inst], pyp + (size_t)inst * MPCB_NPYP,
               pymp + (size_t)inst * MPCB_NPYP, yl);
    for (int i = 0; i < NY; ++i) y[(size_t)inst * NY + i] = yl[i] + (noise ? noise[(size_t)inst * NY + i] : 0.0);
}
__global__ void k_plant_step(int B, double* x, const double* u, const double* t, const double* pxp, const double* pxmp) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    plant_step(x + (size_t)inst * MPCB_NXP, u + (size_t)inst * NU, t[inst], pxp + (size_t)inst * MPCB_NPXP,
               pxmp + (size_t)inst * MPCB_NPXP);
}
#endif


#if MPCB_HAS_OCP && MPCB_HAS_TARGET
// ---------------------------------------------------------------------------------------------
// Loop glue of one closed-loop step as device kernels (mpcb_step): the statements of MPC_code.py:655-700,
// 714-718, 734-772 and 786-805 for every instance.
// ---------------------------------------------------------------------------------------------
struct LoopState {      // per-instance loop state kept on the device between steps (MPC_code.py:442-463)
    double *xi, *P, *u, *us, *xs, *wguess, *wopt, *x0m, *u0, *parss, *wss, *par, *w, *px0, *py0, *fss;
    int *dyn_status, *ss_status, *ss_iters;
};

__global__ void k_step_params(int B, const double* px, const double* py, LoopState L) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    for (int i = 0; i < NPX; ++i) L.px0[(size_t)inst * NPX + i] = px ? px[(size_t)inst * NPX * NH + i] : 0.0;
    for (int i = 0; i < NPY; ++i) L.py0[(size_t)inst * NPY + i] = py ? py[(size_t)inst * NPY * NH + i] : 0.0;
}

// after the estimator: outputs, par_ss (Target_Calc.py:41-50 order, MPC_code.py:693) and the target guess (:696-700)
__global__ void k_step_pre(int B, const double* t, const double* sp, LoopState L, double* xhat_out, double* dhat_out) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= B) return;
    const double* xi = L.xi + (size_t)inst * NXI;
    double* ps = L.parss + (size_t)inst * MPCB_NPARSS;
    for (int i = 0; i < NX; ++i) xhat_out[(size_t)inst * NX + i] = xi[i];
    double d[ND + 1];
    for (int i = 0; i < ND; ++i) { d[i] = (NXI > NX) ? xi[NX + i] : 0.0; dhat_out[(size_t)inst * ND + i] = d[i]; }
    const double* spi = sp + (size_t)inst * (NU + NY + NX);
    for (int i = 0; i < NU; ++i) ps[MPCB_OFFSS_USP + i] = spi[i];
    for (int i = 0; i < NY; ++i) ps[MPCB_OFFSS_YSP + i] = spi[NU + i];
    for (int i = 0; i < NX; ++i) ps[MPCB_OFFSS_XSP + i] = spi[NU + NY + i];
    for (int i = 0; i < ND; ++i) ps[MPCB_OFFSS_D + i] = d[i];
    for (int i = 0; i < NU; ++i) ps[MPCB_OFFSS_USPREV + i] = L.us[(size_t)inst * NU + i];
    for (int i = 0; i < NY * NU; ++i) ps[MPCB_OFFSS_LAM + i] = 0.0;
    ps[MPCB_OFFSS_T] = t[inst];
    double py[NPY + 1];
    for (int i = 0; i < NPX; ++i) ps[MPCB_OFFSS_PX + i] = L.px0[(size_t)inst * NPX + i];
    for (int i = 0; i < NPY; ++i) { py[i] = L.py0[(size_t)inst * NPY + i]; ps[MPCB_OFFSS_PY + i] = py[i]; }
    double* wg = L.wss + (size_t)inst * NWS;
    double x0[NX], u0[NU], y0[NY], tt = t[inst];
    for (int i = 0; i < NX; ++i) { x0[i] = L.x0m[(size_t)inst * NX + i]; wg[i] = x0[i]; }
    for (int i = 0; i < NU; ++i) { u0[i] = L.u0[(size_t)inst * NU + i]; wg[NX + i] = u0[i]; }
    mdl_fy(x0, u0, d, &tt, py, y0);
    for (int i = 0; i < NY; ++i) wg[NZ + i] = y0[i];
}

// after the target solve: status gate (:714-718), par (Control_Calc.py:43-57 order, MPC_code.py:769-772), warm start (:740-764)
// One WARP per instance: the bulk of the work is moving the NW-long iterate (shifted warm start) and the parameter
// rows, which lanes do with coalesced strided copies; one thread per instance spent 0.2 ms per step on serial copies.
__global__ void k_step_mid(int B, int first, const double* t, const double* px, const double* py, LoopState L,
                           double* xs_out, double* us_out) {
    const int inst = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (inst >= B) return;
    double* xs = L.xs + (size_t)inst * NX; double* us = L.us + (size_t)inst * NU;
    const double* wss = L.wss + (size_t)inst * NWS;
    const bool ss_ok = L.ss_status[inst] != 2;
    double xs_prev[NX], us_prev[NU], xs_new[NX], us_new[NU];
    for (int i = 0; i < NX; ++i) { xs_prev[i] = xs[i]; xs_new[i] = ss_ok ? wss[i] : xs_prev[i]; }
    for (int i = 0; i < NU; ++i) { us_prev[i] = us[i]; us_new[i] = ss_ok ? wss[NX + i] : us_prev[i]; }
    __syncwarp();
    const double* xi = L.xi + (size_t)inst * NXI;
    double* pr = L.par + (size_t)inst * NPAR;
    if (lane == 0) {
        for (int i = 0; i < NX; ++i) { xs[i] = xs_new[i]; xs_out[(size_t)inst * NX + i] = xs_new[i]; }
        for (int i = 0; i < NU; ++i) { us[i] = us_new[i]; us_out[(size_t)inst * NU + i] = us_new[i]; }
        for (int i = 0; i < NX; ++i) { pr[MPCB_OFF_X0 + i] = xi[i]; pr[MPCB_OFF_XS + i] = xs_new[i]; }
        for (int i = 0; i < NU; ++i) { pr[MPCB_OFF_US + i] = us_new[i]; pr[MPCB_OFF_UM1 + i] = L.u[(size_t)inst * NU + i]; }
        for (int i = 0; i < ND; ++i) pr[MPCB_OFF_D + i] = (NXI > NX) ? xi[NX + i] : 0.0;
        pr[MPCB_OFF_T] = t[inst];
        for (int i = 0; i < NY * NU; ++i) pr[MPCB_OFF_LAM + i] = 0.0;
    }
    for (int i = lane; i < NPX * NH; i += 32) pr[MPCB_OFF_PX + i] = px ? px[(size_t)inst * NPX * NH + i] : 0.0;
    for (int i = lane; i < NPY * NH; i += 32) pr[MPCB_OFF_PY + i] = py ? py[(size_t)inst * NPY * NH + i] : 0.0;
    double* wg = L.wguess + (size_t)inst * NW; double* w = L.w + (size_t)inst * NW;
    const double* wo = L.wopt + (size_t)inst * NW;
    const bool shift = !first && L.dyn_status[inst] != 2 && L.dyn_status[inst] != -13;
    for (int i = lane; i < NW; i += 32) {
        double v;
        if (first) {
            const int r = i % NZ;
            v = (r < NX) ? L.x0m[(size_t)inst * NX + r] : L.u0[(size_t)inst * NU + r - NX];
        } else if (shift) {
            if (i < NW - NZ) v = wo[NZ + i];
            else {
                v = 0.0;
#pragma unroll
                for (int j = 0; j < NU; ++j) if (i == NW - NZ + j) v = us_prev[j];
#pragma unroll
                for (int j = 0; j < NX; ++j) if (i == NW - NX + j) v = xs_prev[j];
            }
        } else {
            v = wg[i];
        }
        wg[i] = v; w[i] = v;
    }
}

// after the OCP: status gate, u_k and x(k+1|k) extraction or model fallback (:786-805); one warp per instance
// hold_failed: treat every failed solve (status < 0: iteration limit, restoration failed, step computation) like an
// infeasible one - keep the previous input and propagate the estimate with the model.  The reference applies such
// iterates to the plant (only 'Infeasible_Problem_Detected' is rejected, MPC_code.py:786); that stays the default.
__global__ void k_step_post(int B, const double* t, const int* status, LoopState L, double* u_out, int hold_failed) {
    const int inst = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (inst >= B) return;
    double* xi = L.xi + (size_t)inst * NXI; double* u = L.u + (size_t)inst * NU;
    const double* w = L.w + (size_t)inst * NW;
    int st = status[inst];
    if (hold_failed && st < 0 && st != -13) st = 2;
    if (lane == 0) L.dyn_status[inst] = st;
    if (st == -13) {                                      // diverged instance (NaN state): frozen, u keeps its value
        for (int i = lane; i < NU; i += 32) u_out[(size_t)inst * NU + i] = u[i];
    } else if (st != 2) {
        double* wo = L.wopt + (size_t)inst * NW;
        for (int i = lane; i < NW; i += 32) wo[i] = w[i];
        for (int i = lane; i < NU; i += 32) { const double v = w[NX + i]; u[i] = v; u_out[(size_t)inst * NU + i] = v; }
        for (int i = lane; i < NX; i += 32) xi[i] = w[NZ + i];
    } else if (lane == 0) {
        double x[NX], ul[NU], d[ND + 1], pxl[NPX + 1], xn[NX];
        for (int i = 0; i < NX; ++i) x[i] = xi[i];
        for (int i = 0; i < NU; ++i) { ul[i] = u[i]; u_out[(size_t)inst * NU + i] = ul[i]; }
        for (int i = 0; i < ND; ++i) d[i] = (NXI > NX) ? xi[NX + i] : 0.0;
        for (int i = 0; i < NPX; ++i) pxl[i] = L.px0[(size_t)inst * NPX + i];
        dyn_value(x, ul, d, pxl, t[inst], xn);
        for (int i = 0; i < NX; ++i) xi[i] = xn[i];
    }
}
#endif

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct mpcb_ctx {
    int B, device;
    mpcb_opts_t opts_ss, opts_dyn;
    std::string err;
    double *ws, *lbx, *ubx, *lbg, *ubg, *ss_lbx, *ss_ubx, *Qkf, *Rkf, *Kest, *dmin, *dmax;
    InstState* st;
    int* n_active; int* h_active;
    int have_dbounds, last_launches, last_ticks;
    // device-driven solve: a CUDA graph [init -> WHILE {eval, kkt, trial, accept, cond} -> output], rebuilt when the
    // caller's buffers or the options change; tick counters on the device; launches made from the host so far
    cudaGraph_t og_graph; cudaGraphExec_t og_exec;
    const void* og_key[5]; mpcb_opts_t og_opts; int og_valid;
    double* stage_mem; int* stage_imem;      // staging copies of par | w | f and status | iters for callers whose buffers move
    unsigned long long* tick_ctr;            // device: {ticks of the last solve, ticks since creation}
    long host_launches; int host_loop; cudaStream_t last_stream;
    int hold_failed;                         // mpcb_set_policy
    // loop state of the fused step (mpcb_loop_reset / mpcb_step)
    double* loop_mem; int* loop_imem; int loop_first;
#if MPCB_HAS_OCP && MPCB_HAS_TARGET
    LoopState L;
#endif
    // profiling (mpcb_set_profiling): CUDA-event time and launch count per kernel class
    int profile;
    unsigned long long* counters;
    double kernel_ms[MPCB_NKERNELS]; long kernel_launches[MPCB_NKERNELS];
    unsigned long long eval_instances, trial_instances;
    std::vector<cudaEvent_t> ev_pool;
    std::vector<std::pair<int, int>> ev_pending;   // (kernel class, index of start event; stop = +1)
    // instance groups of the fused step (mpcb_set_groups): sub-batches queued on their own streams
    int ngroups;
    std::vector<struct StepGroup*> groups;
    cudaEvent_t ev_in;
};

struct StepGroup { mpcb_ctx* c; int b0, nb; cudaStream_t s; cudaEvent_t done; };

static IpmOpts to_ipm(const mpcb_opts_t& o) {
    IpmOpts r;
    r.max_iter = o.max_iter; r.tol = o.tol; r.mu_init = o.mu_init; r.bound_relax = o.bound_relax_factor;
    r.bound_push = o.bound_push; r.acceptable_tol = o.acceptable_tol;
    r.honor_original_bounds = o.honor_original_bounds; r.acceptable_iter = o.acceptable_iter;
    return r;
}

static int fail(mpcb_ctx* h, const char* what, cudaError_t e) {
    if (h) h->err = std::string(what) + ": " + cudaGetErrorString(e);
    return -1;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(h, #call, e_); } while (0)

// Launch bracket: with profiling on, a pair of events goes around the launch on its own stream.
struct Prof {
    mpcb_ctx* h; cudaStream_t s; int kc; int idx;
    Prof(mpcb_ctx* h_, cudaStream_t s_, int kc_) : h(h_), s(s_), kc(kc_), idx(-1) {
        if (!h->profile) return;
        idx = (int)h->ev_pending.size() * 2;
        while ((int)h->ev_pool.size() < idx + 2) { cudaEvent_t e; cudaEventCreate(&e); h->ev_pool.push_back(e); }
        cudaEventRecord(h->ev_pool[idx], s);
    }
    ~Prof() {
        h->kernel_launches[kc] += 1;
        if (idx < 0) return;
        cudaEventRecord(h->ev_pool[idx + 1], s);
        h->ev_pending.push_back(std::make_pair(kc, idx));
    }
};
static void prof_collect(mpcb_ctx* h) {       // call after the stream has been synchronised
    for (auto& p : h->ev_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->ev_pool[p.second], h->ev_pool[p.second + 1]) == cudaSuccess) h->kernel_ms[p.first] += ms;
    }
    h->ev_pending.clear();
}

__global__ void k_dfma_peak(double* out, int iters) {
    // 8 independent FMA chains per thread: measures the FP64 FMA issue rate of the part
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double b = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

extern "C" {

int mpcb_abi_version(void) { return MPCB_ABI_VERSION; }

void mpcb_default_opts(mpcb_opts_t* o) {
    o->max_iter = 100; o->tol = 1e-8; o->mu_init = 0.1; o->bound_relax_factor = 1e-8;
    o->honor_original_bounds = 0; o->bound_push = 1e-2; o->acceptable_tol = 1e-6; o->acceptable_iter = 15;
}

int mpcb_get_dims(mpcb_dims_t* d) {
    memset(d, 0, sizeof(*d));
    d->nx = NX; d->nu = NU; d->ny = NY; d->nd = ND; d->npx = NPX; d->npy = NPY;
    d->nxp = MPCB_NXP; d->npxp = MPCB_NPXP; d->npyp = MPCB_NPYP; d->nxi = NXI; d->N = NH; d->Mx = MX;
#if MPCB_HAS_OCP
    d->nw = NW; d->npar = NPAR; d->ng = NG; d->has_ocp = 1;
#endif
#if MPCB_HAS_TARGET
    d->nwss = NWS; d->nparss = MPCB_NPARSS; d->has_target = 1;
#endif
    return 0;
}

long mpcb_model_flops(const char* name) {
    static const struct { const char* n; long f; } table[] = { MPCB_FLOPS_TABLE {nullptr, 0} };
    for (int i = 0; table[i].n; ++i) if (!strcmp(table[i].n, name)) return table[i].f;
    return -1;
}

int mpcb_create(int batch, const mpcb_opts_t* oss, const mpcb_opts_t* odyn, mpcb_handle_t* out) {
    mpcb_ctx* h = new mpcb_ctx();
    h->B = batch; h->have_dbounds = 0; h->last_launches = 0; h->last_ticks = 0;
    h->og_graph = nullptr; h->og_exec = nullptr; h->og_valid = 0; h->tick_ctr = nullptr; h->host_launches = 0; h->last_stream = nullptr;
    h->stage_mem = nullptr; h->stage_imem = nullptr; h->hold_failed = 0;
    { const char* e = getenv("MPCB_HOST_LOOP"); h->host_loop = (e && e[0] == '1') ? 1 : 0; }
    mpcb_default_opts(&h->opts_ss); mpcb_default_opts(&h->opts_dyn);
    if (oss) h->opts_ss = *oss;
    if (odyn) h->opts_dyn = *odyn;
    *out = h;
    if (batch <= 0) { h->err = "batch must be positive"; return -2; }
    CK(cudaGetDevice(&h->device));
    h->ws = nullptr; h->st = nullptr; h->lbx = h->ubx = h->lbg = h->ubg = nullptr;
#if MPCB_HAS_OCP
    CK(cudaMalloc(&h->ws, sizeof(double) * (size_t)batch * OcpLayout::total));
    CK(cudaMemset(h->ws, 0, sizeof(double) * (size_t)batch * OcpLayout::total));
    CK(cudaMalloc(&h->st, sizeof(InstState) * (size_t)batch));
    CK(cudaMalloc(&h->lbx, sizeof(double) * NWI)); CK(cudaMalloc(&h->ubx, sizeof(double) * NWI));
    CK(cudaMalloc(&h->lbg, sizeof(double) * (NH * NGS))); CK(cudaMalloc(&h->ubg, sizeof(double) * (NH * NGS)));
    if (EVAL_SMEM_BYTES > 0) {
        CK(cudaFuncSetAttribute(k_ocp_eval, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EVAL_SMEM_BYTES));
        CK(cudaFuncSetAttribute(k_stage_derivs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EVAL_SMEM_BYTES));
    }
#endif
    h->ss_lbx = h->ss_ubx = nullptr;
#if MPCB_HAS_TARGET
    CK(cudaMalloc(&h->ss_lbx, sizeof(double) * NWS)); CK(cudaMalloc(&h->ss_ubx, sizeof(double) * NWS));
#endif
    CK(cudaMalloc(&h->Qkf, sizeof(double) * NXI * NXI)); CK(cudaMalloc(&h->Rkf, sizeof(double) * NY * NY));
    CK(cudaMalloc(&h->Kest, sizeof(double) * NXI * NY));
    CK(cudaMalloc(&h->dmin, sizeof(double) * (ND + 1))); CK(cudaMalloc(&h->dmax, sizeof(double) * (ND + 1)));
    CK(cudaMemset(h->Qkf, 0, sizeof(double) * NXI * NXI)); CK(cudaMemset(h->Rkf, 0, sizeof(double) * NY * NY));
    CK(cudaMemset(h->Kest, 0, sizeof(double) * NXI * NY));
    CK(cudaMalloc(&h->n_active, sizeof(int)));
    CK(cudaMemset(h->n_active, 0, sizeof(int)));
    CK(cudaMallocHost(&h->h_active, sizeof(int)));
    CK(cudaMalloc(&h->tick_ctr, 2 * sizeof(unsigned long long)));
    CK(cudaMemset(h->tick_ctr, 0, 2 * sizeof(unsigned long long)));
    CK(cudaMalloc(&h->counters, 2 * sizeof(unsigned long long)));
    CK(cudaMemset(h->counters, 0, 2 * sizeof(unsigned long long)));
    h->loop_mem = nullptr; h->loop_imem = nullptr; h->loop_first = 1;
    h->profile = 0; h->eval_instances = h->trial_instances = 0;
    h->ngroups = 1; h->ev_in = nullptr;
    for (int i = 0; i < MPCB_NKERNELS; ++i) { h->kernel_ms[i] = 0.0; h->kernel_launches[i] = 0; }
    return 0;
}

static void groups_teardown(mpcb_ctx* h);

static void ocp_graph_drop(mpcb_ctx* h) {
    if (h->og_exec) cudaGraphExecDestroy(h->og_exec);
    if (h->og_graph) cudaGraphDestroy(h->og_graph);
    h->og_exec = nullptr; h->og_graph = nullptr; h->og_valid = 0;
}

int mpcb_destroy(mpcb_handle_t h) {
    if (!h) return 0;
    cudaDeviceSynchronize();
    groups_teardown(h);
    ocp_graph_drop(h);
    cudaFree(h->tick_ctr); cudaFree(h->stage_mem); cudaFree(h->stage_imem);
    if (h->ev_in) cudaEventDestroy(h->ev_in);
    cudaFree(h->ws); cudaFree(h->st); cudaFree(h->lbx); cudaFree(h->ubx); cudaFree(h->lbg); cudaFree(h->ubg);
    cudaFree(h->ss_lbx); cudaFree(h->ss_ubx); cudaFree(h->Qkf); cudaFree(h->Rkf); cudaFree(h->Kest);
    cudaFree(h->dmin); cudaFree(h->dmax); cudaFree(h->n_active); cudaFreeHost(h->h_active); cudaFree(h->counters);
    for (auto e : h->ev_pool) cudaEventDestroy(e);
    cudaFree(h->loop_mem); cudaFree(h->loop_imem);
    delete h;
    return 0;
}

const char* mpcb_last_error(mpcb_handle_t h) { return h ? h->err.c_str() : "null handle"; }

int mpcb_set_const(mpcb_handle_t h, const char* name, const double* p, int n) {
#if MPCB_HAS_OCP
    if (!strcmp(name, "ocp_lbx") || !strcmp(name, "ocp_ubx")) {
        // reference layout [x0,u0,...,xN] -> internal layout [z0,u0,...,zN], z = [x; v]; the carried inputs v are free
        if (n != NW) { h->err = std::string("mpcb_set_const: wrong length for ") + name; return -2; }
        const bool lower = !strcmp(name, "ocp_lbx");
        std::vector<double> tmp(NWI, lower ? -INFINITY : INFINITY);
        for (int k = 0; k <= NH; ++k) {
            for (int i = 0; i < NX; ++i) tmp[k * NZA + i] = p[k * NZ + i];
            if (k < NH) for (int i = 0; i < NU; ++i) tmp[k * NZA + NXA + i] = p[k * NZ + NX + i];
        }
        CK(cudaMemcpy(lower ? h->lbx : h->ubx, tmp.data(), sizeof(double) * NWI, cudaMemcpyHostToDevice));
        return 0;
    }
#endif
    struct { const char* nm; double* dst; int len; } tab[] = {
#if MPCB_HAS_OCP
        {"ocp_lbg", h->lbg, NH * NG}, {"ocp_ubg", h->ubg, NH * NG},
#endif
#if MPCB_HAS_TARGET
        {"ss_lbx", h->ss_lbx, NWS}, {"ss_ubx", h->ss_ubx, NWS},
#endif
        {"Q_kf", h->Qkf, NXI * NXI}, {"R_kf", h->Rkf, NY * NY}, {"K_est", h->Kest, NXI * NY},
        {"dmin", h->dmin, ND}, {"dmax", h->dmax, ND},
    };
    for (auto& e : tab) {
        if (strcmp(e.nm, name)) continue;
        if (n != e.len) { h->err = std::string("mpcb_set_const: wrong length for ") + name; return -2; }
        if (n > 0) CK(cudaMemcpy(e.dst, p, sizeof(double) * n, cudaMemcpyHostToDevice));
        if (!strcmp(name, "dmax")) h->have_dbounds = 1;
        return 0;
    }
    h->err = std::string("mpcb_set_const: unknown name ") + name;
    return -2;
}

static inline int nblk(long n, int bs) { return (int)((n + bs - 1) / bs); }

static bool same_opts(const mpcb_opts_t& a, const mpcb_opts_t& b) {
    return a.max_iter == b.max_iter && a.tol == b.tol && a.mu_init == b.mu_init && a.bound_relax_factor == b.bound_relax_factor &&
           a.honor_original_bounds == b.honor_original_bounds && a.bound_push == b.bound_push &&
           a.acceptable_tol == b.acceptable_tol && a.acceptable_iter == b.acceptable_iter;
}

#if MPCB_HAS_OCP
// Build the device-driven solve as a CUDA graph:
//   memset counters -> k_ocp_init -> U unrolled ticks -> k_ocp_cond -> WHILE { tick -> k_ocp_cond } -> k_ocp_output
// with tick = k_ocp_eval -> k_ocp_kkt -> k_ocp_trial -> k_ocp_accept.  The loop condition is set on the device by k_ocp_cond
// (cudaGraphSetConditional), so a whole solve - however many ticks its slowest instance needs - is ONE graph launch and the
// host never waits on it (round 1 polled a device counter every two ticks, with one spinning host thread per group).
// The first U ticks are plain kernel nodes: a node inside a WHILE body costs ~5 us of device-side scheduling that
// serialises across streams (measured: profiles/r02_groups_sweep_graph.txt), a plain node ~1.5 us, and a tick whose
// instances are all done is four kernels that exit at once.  U = MPCB_GRAPH_UNROLL (environment), default 10: a warm
// closed-loop step of Ex_NMPC needs 11-13 ticks.
#define TICK_KERNELS 4                   // launches per tick
static int add_tick(mpcb_ctx* h, cudaGraph_t g, cudaGraphNode_t* dep, int ndep, OcpArgs& a, int* n_active, cudaGraphNode_t* last,
                    bool first = false) {
    const int bs = 128;
    const long nst = (long)h->B * NH;
    cudaKernelNodeParams kp; memset(&kp, 0, sizeof(kp));
    void* args1[] = {&a};
    cudaGraphNode_t n_eval;
    kp.kernelParams = args1;
    kp.func = (void*)k_ocp_eval; kp.gridDim = dim3(nblk(nst, MPCB_EVAL_BLOCK)); kp.blockDim = dim3(MPCB_EVAL_BLOCK);
    kp.sharedMemBytes = (unsigned)EVAL_SMEM_BYTES;
#if MPCB_EVAL_FIRST
    if (first) { kp.func = (void*)k_ocp_eval_first; kp.gridDim = dim3(nblk(nst, 128)); kp.blockDim = dim3(128); kp.sharedMemBytes = 0; }
#else
    (void)first;
#endif
    CK(cudaGraphAddKernelNode(&n_eval, g, dep, ndep, &kp));
    kp.sharedMemBytes = 0;
    { dim3 gk(1), bk(1); auto set = [&](int gx, int bx) { gk = dim3(gx); bk = dim3(bx); }; set(KKT_GRID(h->B));
      kp.func = (void*)k_ocp_kkt; kp.gridDim = gk; kp.blockDim = bk; }
    cudaGraphNode_t n_kkt, n_trial;
    CK(cudaGraphAddKernelNode(&n_kkt, g, &n_eval, 1, &kp));
    kp.func = (void*)k_ocp_trial; kp.gridDim = dim3(nblk(nst, bs)); kp.blockDim = dim3(bs);
    CK(cudaGraphAddKernelNode(&n_trial, g, &n_kkt, 1, &kp));
    void* args2[] = {&a, &n_active};
    kp.func = (void*)k_ocp_accept; kp.gridDim = dim3(nblk((long)h->B * 32, 32 * KKT_WARPS)); kp.blockDim = dim3(32 * KKT_WARPS);
    kp.kernelParams = args2;
    CK(cudaGraphAddKernelNode(last, g, &n_trial, 1, &kp));
    return 0;
}

static int ocp_graph_build(mpcb_ctx* h, const OcpArgs& a_in, double* f, int* status, int* iters) {
    ocp_graph_drop(h);
    OcpArgs a = a_in;
    const int bs = 128;
    int max_ticks = (h->opts_dyn.max_iter + 2) * 8;
    int unroll = 10;
    { const char* e = getenv("MPCB_GRAPH_UNROLL"); if (e) unroll = atoi(e); }
    if (unroll < 0) unroll = 0;
    if (unroll > max_ticks) unroll = max_ticks;
    CK(cudaGraphCreate(&h->og_graph, 0));
    cudaGraph_t g = h->og_graph;
    cudaGraphNode_t n_ms1, n_ms2, n_init, n_while, n_out, prev;
    cudaMemsetParams ms; memset(&ms, 0, sizeof(ms));
    ms.dst = h->n_active; ms.value = 0; ms.elementSize = 4; ms.width = 1; ms.height = 1; ms.pitch = 4;
    CK(cudaGraphAddMemsetNode(&n_ms1, g, nullptr, 0, &ms));
    ms.dst = h->tick_ctr; ms.width = 2;                                 // ticks of this solve (one 64-bit counter)
    CK(cudaGraphAddMemsetNode(&n_ms2, g, nullptr, 0, &ms));
    cudaKernelNodeParams kp; memset(&kp, 0, sizeof(kp));
    void* args1[] = {&a};
    kp.func = (void*)k_ocp_init; kp.gridDim = dim3(nblk((long)h->B * (NH + 1), bs)); kp.blockDim = dim3(bs); kp.kernelParams = args1;
    cudaGraphNode_t dep0[] = {n_ms1, n_ms2};
    CK(cudaGraphAddKernelNode(&n_init, g, dep0, 2, &kp));
    prev = n_init;
    int* n_active = h->n_active; int* no_count = nullptr;
    for (int t = 0; t < unroll; ++t) {                                   // only the last unrolled tick counts the active instances
        cudaGraphNode_t last;
        int rc = add_tick(h, g, &prev, 1, a, (t == unroll - 1) ? n_active : no_count, &last, t == 0);
        if (rc) return rc;
        prev = last;
    }
    cudaGraphConditionalHandle handle;
    CK(cudaGraphConditionalHandleCreate(&handle, g, 1, cudaGraphCondAssignDefault));
    unsigned long long* ctr = h->tick_ctr;
    if (unroll > 0) {                                                    // condition for entering the WHILE tail
        cudaGraphNode_t n_c0;
        void* args3[] = {&handle, &n_active, &ctr, &max_ticks, &unroll};
        kp.func = (void*)k_ocp_cond; kp.gridDim = dim3(1); kp.blockDim = dim3(1); kp.kernelParams = args3; kp.sharedMemBytes = 0;
        CK(cudaGraphAddKernelNode(&n_c0, g, &prev, 1, &kp));
        prev = n_c0;
    }
    cudaGraphNodeParams cp = { cudaGraphNodeTypeConditional };
    cp.conditional.handle = handle; cp.conditional.type = cudaGraphCondTypeWhile; cp.conditional.size = 1;
    CK(cudaGraphAddNode(&n_while, g, &prev, 1, &cp));
    cudaGraph_t body = cp.conditional.phGraph_out[0];
    {
        cudaGraphNode_t last, n_cond;
        int rc = add_tick(h, body, nullptr, 0, a, n_active, &last);
        if (rc) return rc;
        int one = 1;
        void* args3[] = {&handle, &n_active, &ctr, &max_ticks, &one};
        kp.func = (void*)k_ocp_cond; kp.gridDim = dim3(1); kp.blockDim = dim3(1); kp.kernelParams = args3; kp.sharedMemBytes = 0;
        CK(cudaGraphAddKernelNode(&n_cond, body, &last, 1, &kp));
    }
    void* args4[] = {&a, &f, &status, &iters};
    kp.func = (void*)k_ocp_output; kp.gridDim = dim3(nblk((long)h->B * (NH + 1), 128)); kp.blockDim = dim3(128); kp.kernelParams = args4;
    CK(cudaGraphAddKernelNode(&n_out, g, &n_while, 1, &kp));
    CK(cudaGraphInstantiate(&h->og_exec, g, 0));
    h->og_key[0] = a.par; h->og_key[1] = a.w; h->og_key[2] = f; h->og_key[3] = status; h->og_key[4] = iters;
    h->og_opts = h->opts_dyn; h->og_valid = 1;
    return 0;
}

// host-polled variant of the same schedule: used with profiling on (event brackets around every launch) or MPCB_HOST_LOOP=1
static int ocp_host_loop(mpcb_ctx* h, OcpArgs& a, double* f, int* status, int* iters, cudaStream_t s) {
    const int bs = 128;
    const long nst = (long)h->B * NH;
    int launches = 0, ticks = 0;
    CK(cudaMemsetAsync(h->n_active, 0, sizeof(int), s));
    { Prof p(h, s, KC_OCP_INIT); k_ocp_init<<<nblk((long)h->B * (NH + 1), bs), bs, 0, s>>>(a); } launches++;
    // every instance needs at most max_iter+1 evaluations plus its line-search backtracks
    const int max_ticks = (h->opts_dyn.max_iter + 2) * 8;
    const int check_every = 2;
    while (ticks < max_ticks) {
        for (int c = 0; c < check_every; ++c) {
#if MPCB_EVAL_FIRST
            if (ticks == 0) { Prof p(h, s, KC_OCP_EVAL); k_ocp_eval_first<<<nblk(nst, 128), 128, 0, s>>>(a); }
            else
#endif
            { Prof p(h, s, KC_OCP_EVAL); k_ocp_eval<<<nblk(nst, MPCB_EVAL_BLOCK), MPCB_EVAL_BLOCK, EVAL_SMEM_BYTES, s>>>(a); }
            { Prof p(h, s, KC_OCP_KKT); k_ocp_kkt<<<KKT_GRID(h->B), 0, s>>>(a); }
            { Prof p(h, s, KC_OCP_TRIAL); k_ocp_trial<<<nblk(nst, bs), bs, 0, s>>>(a); }
            if (c == check_every - 1) CK(cudaMemsetAsync(h->n_active, 0, sizeof(int), s));
            { Prof p(h, s, KC_OCP_ACCEPT); k_ocp_accept<<<nblk((long)h->B * 32, 32 * KKT_WARPS), 32 * KKT_WARPS, 0, s>>>(a, h->n_active); }
            launches += TICK_KERNELS; ticks++;
        }
        CK(cudaMemcpyAsync(h->h_active, h->n_active, sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        prof_collect(h);
        if (*h->h_active == 0) break;
    }
    CK(cudaMemsetAsync(h->n_active, 0, sizeof(int), s));
    { Prof p(h, s, KC_OTHER); k_ocp_output<<<nblk((long)h->B * (NH + 1), 128), 128, 0, s>>>(a, f, status, iters); } launches++;
    CK(cudaGetLastError());
    if (h->profile) {
        unsigned long long cnt[2];
        CK(cudaMemcpyAsync(cnt, h->counters, sizeof(cnt), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        prof_collect(h);
        h->eval_instances = cnt[0]; h->trial_instances = cnt[1];
    }
    h->host_launches += launches;
    h->last_launches = launches; h->last_ticks = ticks;
    return 0;
}
#endif

// Asynchronous: the solve is queued on `stream` (one CUDA-graph launch) and the call returns; outputs are complete when
// the stream reaches that point.  With profiling on it runs the host-polled schedule and returns after completion.
int mpcb_ocp(mpcb_handle_t h, const double* par, double* w, double* f, int* status, int* iters, void* stream) {
#if MPCB_HAS_OCP
    cudaStream_t s = (cudaStream_t)stream;
    OcpArgs a;
    a.B = h->B; a.par = par; a.w = w; a.ws = h->ws; a.st = h->st; a.counters = h->counters;
    a.S.lbx = h->lbx; a.S.ubx = h->ubx; a.S.lbg = h->lbg; a.S.ubg = h->ubg; a.S.o = to_ipm(h->opts_dyn);
    h->last_stream = s;
    if (h->profile || h->host_loop) return ocp_host_loop(h, a, f, status, iters, s);
    // The graph holds its buffers' addresses.  A caller whose buffers stay put (the fused step; any caller that reuses its
    // tensors) is served in place; one whose buffers move gets staging copies from its second call on, so that the graph
    // is built once, not per call.
    const void* key[5] = {par, w, f, status, iters};
    const bool moved = h->og_valid && memcmp(key, h->og_key, sizeof(key)) != 0;
    const size_t B = (size_t)h->B;
    if (moved && !h->stage_mem) {
        CK(cudaMalloc(&h->stage_mem, sizeof(double) * B * (NPAR + NW + 1)));
        CK(cudaMalloc(&h->stage_imem, sizeof(int) * B * 2));
    }
    const bool staged = h->stage_mem != nullptr;
    double* sp_ = h->stage_mem; double* sw_ = sp_ + B * NPAR; double* sf_ = sw_ + B * NW;
    int* sst_ = h->stage_imem; int* sit_ = sst_ + B;
    if (staged) {
        CK(cudaMemcpyAsync(sp_, par, sizeof(double) * B * NPAR, cudaMemcpyDeviceToDevice, s));
        CK(cudaMemcpyAsync(sw_, w, sizeof(double) * B * NW, cudaMemcpyDeviceToDevice, s));
        a.par = sp_; a.w = sw_;
        key[0] = sp_; key[1] = sw_; key[2] = sf_; key[3] = sst_; key[4] = sit_;
    }
    if (!h->og_valid || memcmp(key, h->og_key, sizeof(key)) || !same_opts(h->og_opts, h->opts_dyn)) {
        int rc = staged ? ocp_graph_build(h, a, sf_, sst_, sit_) : ocp_graph_build(h, a, f, status, iters);
        if (rc) return rc;
    }
    CK(cudaGraphLaunch(h->og_exec, s));
    if (staged) {
        CK(cudaMemcpyAsync(w, sw_, sizeof(double) * B * NW, cudaMemcpyDeviceToDevice, s));
        CK(cudaMemcpyAsync(f, sf_, sizeof(double) * B, cudaMemcpyDeviceToDevice, s));
        CK(cudaMemcpyAsync(status, sst_, sizeof(int) * B, cudaMemcpyDeviceToDevice, s));
        CK(cudaMemcpyAsync(iters, sit_, sizeof(int) * B, cudaMemcpyDeviceToDevice, s));
    }
    h->host_launches += 2;                       // init + output; the ticks are counted on the device (4-5 launches each)
    h->last_launches = -1; h->last_ticks = -1;   // known once the stream has run: see mpcb_last_ticks
    return 0;
#else
    h->err = "library built without the OCP"; return -3;
#endif
}

long mpcb_ocp_sens_size(void) {
#if MPCB_HAS_OCP
    return SensLayout::total;
#else
    return 0;
#endif
}

// Reads the workspace of the handle's last mpcb_ocp (records, iterate, multipliers, per-instance status) and writes
// only `fac` and `status`: the next solve starts from k_ocp_init exactly as without this call.
int mpcb_ocp_sens_factor(mpcb_handle_t h, const double* par, double* fac, int* status, void* stream) {
#if MPCB_HAS_OCP
    cudaStream_t s = (cudaStream_t)stream;
    h->host_launches += 1;
    { Prof p(h, s, KC_OTHER); k_ocp_sens_factor<<<KKT_GRID(h->B), 0, s>>>(h->B, h->ws, par, h->st, fac, status); }
    CK(cudaGetLastError());
    return 0;
#else
    h->err = "library built without the OCP"; return -3;
#endif
}

#if MPCB_HAS_OCP
static int sens_refuse(mpcb_ctx* h) {
    if (!MPCB_SENS_CONT_DEP) return 0;
    h->err = "OCP sensitivities: the ContForm cost integrand depends on the targets / initial state, whose mixed "
             "derivatives through the integrator are not generated";
    return -4;
}
#endif

int mpcb_ocp_jvp(mpcb_handle_t h, const double* fac, int ndir, const double* dtheta, double* dw, void* stream) {
#if MPCB_HAS_OCP
    if (int rc = sens_refuse(h)) return rc;
    if (ndir < 0) { h->err = "mpcb_ocp_jvp: ndir must be >= 0"; return -2; }
    if (ndir == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    h->host_launches += 1;
    { Prof p(h, s, KC_OTHER); k_ocp_jvp<<<nblk((long)h->B * ndir, 128), 128, 0, s>>>(h->B, ndir, fac, dtheta, dw); }
    CK(cudaGetLastError());
    return 0;
#else
    h->err = "library built without the OCP"; return -3;
#endif
}

int mpcb_ocp_vjp(mpcb_handle_t h, const double* fac, const double* gw, double* gtheta, void* stream) {
#if MPCB_HAS_OCP
    if (int rc = sens_refuse(h)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    h->host_launches += 1;
    { Prof p(h, s, KC_OTHER); k_ocp_vjp<<<nblk(h->B, 128), 128, 0, s>>>(h->B, fac, gw, gtheta); }
    CK(cudaGetLastError());
    return 0;
#else
    h->err = "library built without the OCP"; return -3;
#endif
}

long mpcb_ocp_sens_size_p(void) {
#if MPCB_HAS_OCP
    return SensLayout::total + SensPLayout::total;
#else
    return 0;
#endif
}

#if MPCB_HAS_OCP
static int sens_p_refuse(mpcb_ctx* h) {
    if (MPCB_SENS_P) return 0;
    h->err = "OCP sensitivities with respect to d / px / py are not generated for this problem (ContForm, or a large "
             "model on the dense derivative path, or a stage map that reads another stage's px / py)";
    return -4;
}
#endif

int mpcb_ocp_sens_factor_p(mpcb_handle_t h, const double* par, double* fac, int* status, void* stream) {
#if MPCB_HAS_OCP
    if (int rc = sens_p_refuse(h)) return rc;
#if MPCB_SENS_P
    if (int rc = mpcb_ocp_sens_factor(h, par, fac, status, stream)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    h->host_launches += 1;
    { Prof p(h, s, KC_OTHER); k_ocp_sens_pblocks<<<nblk((long)h->B * (NH + 1), 128), 128, 0, s>>>(h->B, h->ws, par, h->st, fac); }
    CK(cudaGetLastError());
#endif
    return 0;
#else
    h->err = "library built without the OCP"; return -3;
#endif
}

int mpcb_ocp_jvp_p(mpcb_handle_t h, const double* fac, int ndir, const double* dp, double* dw, void* stream) {
#if MPCB_HAS_OCP
    if (int rc = sens_p_refuse(h)) return rc;
    if (ndir < 0) { h->err = "mpcb_ocp_jvp_p: ndir must be >= 0"; return -2; }
    if (ndir == 0) return 0;
#if MPCB_SENS_P
    cudaStream_t s = (cudaStream_t)stream;
    h->host_launches += 1;
    { Prof p(h, s, KC_OTHER); k_ocp_jvp_p<<<nblk((long)h->B * ndir, 128), 128, 0, s>>>(h->B, ndir, fac, dp, dw); }
    CK(cudaGetLastError());
#endif
    return 0;
#else
    h->err = "library built without the OCP"; return -3;
#endif
}

int mpcb_ocp_vjp_p(mpcb_handle_t h, const double* fac, const double* gw, double* gp, void* stream) {
#if MPCB_HAS_OCP
    if (int rc = sens_p_refuse(h)) return rc;
#if MPCB_SENS_P
    cudaStream_t s = (cudaStream_t)stream;
    h->host_launches += 1;
    { Prof p(h, s, KC_OTHER); k_ocp_vjp_p<<<nblk(h->B, 128), 128, 0, s>>>(h->B, fac, gw, gp); }
    CK(cudaGetLastError());
#endif
    return 0;
#else
    h->err = "library built without the OCP"; return -3;
#endif
}

int mpcb_stage_derivs(mpcb_handle_t h, const double* par, const double* w, const double* lam,
                      double* A, double* Bm, double* c, double* H, void* stream) {
#if MPCB_HAS_OCP
    h->host_launches += 1;
    { Prof p(h, (cudaStream_t)stream, KC_OTHER); k_stage_derivs<<<nblk((long)h->B * NH, MPCB_EVAL_BLOCK), MPCB_EVAL_BLOCK, EVAL_SMEM_BYTES, (cudaStream_t)stream>>>(h->B, par, w, lam, A, Bm, c, H); }
    CK(cudaGetLastError());
    h->last_launches = 1;
    return 0;
#else
    h->err = "library built without the OCP"; return -3;
#endif
}

int mpcb_target(mpcb_handle_t h, const double* par_ss, double* wss, double* fss, int* status, int* iters, void* stream) {
#if MPCB_HAS_TARGET
    TgtShared S; S.lbx = h->ss_lbx; S.ubx = h->ss_ubx; S.o = to_ipm(h->opts_ss);
    { Prof p(h, (cudaStream_t)stream, KC_TARGET); k_target<<<nblk(h->B, MPCB_TGT_BLOCK), MPCB_TGT_BLOCK, 0, (cudaStream_t)stream>>>(h->B, par_ss, wss, fss, status, iters, S); }
#if !MPCB_DENSE_SH
    { Prof p(h, (cudaStream_t)stream, KC_TARGET); k_target_resto<<<nblk(h->B, MPCB_TGT_BLOCK), MPCB_TGT_BLOCK, 0, (cudaStream_t)stream>>>(h->B, par_ss, wss, fss, status, iters, S); }
    h->host_launches += 1;
#endif
    CK(cudaGetLastError());
    if (h->profile) { CK(cudaStreamSynchronize((cudaStream_t)stream)); prof_collect(h); }
    h->host_launches += 1; h->last_stream = (cudaStream_t)stream;
    h->last_launches = 1; h->last_ticks = 1;
    return 0;
#else
    h->err = "library built without the target problem"; return -3;
#endif
}

long mpcb_target_sens_size(void) {
#if MPCB_SENS_TGT
    return TgtSensLayout::total;
#else
    return -1;
#endif
}

static int tgt_sens_refuse(mpcb_ctx* h) {
    if (!MPCB_HAS_TARGET) { h->err = "library built without the target problem"; return -3; }
    if (MPCB_SENS_TGT) return 0;
    h->err = "target sensitivities are not generated for this problem (a large model on the dense derivative path, or a "
             "map after the RK4 integration that is not affine in d / px)";
    return -4;
}

// Solves the target problem again from wss0 (not modified) and writes only `fac` and `status`.
int mpcb_target_sens_factor(mpcb_handle_t h, const double* par_ss, const double* wss0, double* fac, int* status, void* stream) {
    if (int rc = tgt_sens_refuse(h)) return rc;
#if MPCB_SENS_TGT
    cudaStream_t s = (cudaStream_t)stream;
    TgtShared S; S.lbx = h->ss_lbx; S.ubx = h->ss_ubx; S.o = to_ipm(h->opts_ss);
    { Prof p(h, s, KC_OTHER); k_target_sens<<<nblk(h->B, MPCB_TGT_BLOCK), MPCB_TGT_BLOCK, 0, s>>>(h->B, par_ss, wss0, fac, status, S); }
    { Prof p(h, s, KC_OTHER); k_target_sens_resto<<<nblk(h->B, MPCB_TGT_BLOCK), MPCB_TGT_BLOCK, 0, s>>>(h->B, par_ss, wss0, fac, status, S); }
    h->host_launches += 2;
    CK(cudaGetLastError());
#endif
    return 0;
}

int mpcb_target_jvp(mpcb_handle_t h, const double* fac, int ndir, const double* dth, double* dwss, void* stream) {
    if (int rc = tgt_sens_refuse(h)) return rc;
    if (ndir < 0) { h->err = "mpcb_target_jvp: ndir must be >= 0"; return -2; }
    if (ndir == 0) return 0;
#if MPCB_SENS_TGT
    cudaStream_t s = (cudaStream_t)stream;
    h->host_launches += 1;
    { Prof p(h, s, KC_OTHER); k_target_jvp<<<nblk((long)h->B * ndir, 128), 128, 0, s>>>(h->B, ndir, fac, dth, dwss); }
    CK(cudaGetLastError());
#endif
    return 0;
}

int mpcb_target_vjp(mpcb_handle_t h, const double* fac, const double* gwss, double* gth, void* stream) {
    if (int rc = tgt_sens_refuse(h)) return rc;
#if MPCB_SENS_TGT
    cudaStream_t s = (cudaStream_t)stream;
    h->host_launches += 1;
    { Prof p(h, s, KC_OTHER); k_target_vjp<<<nblk(h->B, 128), 128, 0, s>>>(h->B, fac, gwss, gth); }
    CK(cudaGetLastError());
#endif
    return 0;
}

int mpcb_estimate(mpcb_handle_t h, int est_type, const double* y, const double* u, const double* t, const double* px,
                  const double* py, double* xi, double* P, void* stream) {
    EstShared E; E.Q = h->Qkf; E.R = h->Rkf; E.K = h->Kest; E.dmin = h->dmin; E.dmax = h->dmax; E.has_dbounds = h->have_dbounds;
    { Prof p(h, (cudaStream_t)stream, KC_ESTIMATE); k_estimate<<<nblk(h->B, 64), 64, 0, (cudaStream_t)stream>>>(h->B, est_type, y, u, t, px, py, xi, P, E); }
    CK(cudaGetLastError());
    h->host_launches += 1;
    return 0;
}

int mpcb_model_output(mpcb_handle_t h, const double* x, const double* u, const double* d, const double* t,
                      const double* py, double* y, void* stream) {
    h->kernel_launches[KC_OTHER] += 1; h->host_launches += 1;
    k_model_output<<<nblk(h->B, 128), 128, 0, (cudaStream_t)stream>>>(h->B, x, u, d, t, py, y);
    CK(cudaGetLastError());
    return 0;
}

int mpcb_model_step(mpcb_handle_t h, const double* x, const double* u, const double* d, const double* t,
                    const double* px, double* xn, void* stream) {
    h->kernel_launches[KC_OTHER] += 1; h->host_launches += 1;
    k_model_step<<<nblk(h->B, 128), 128, 0, (cudaStream_t)stream>>>(h->B, x, u, d, t, px, xn);
    CK(cudaGetLastError());
    return 0;
}

int mpcb_plant_meas(mpcb_handle_t h, const double* x, const double* u, const double* t, const double* pyp,
                    const double* pymp, const double* noise, double* y, void* stream) {
#if !MPCB_PLANT_NOMINAL
    h->kernel_launches[KC_OTHER] += 1; h->host_launches += 1;
    k_plant_meas<<<nblk(h->B, 128), 128, 0, (cudaStream_t)stream>>>(h->B, x, u, t, pyp, pymp, noise, y);
    CK(cudaGetLastError());
    return 0;
#else
    h->err = "nominal plant: use mpcb_model_output (MPC_code.py:531-532)"; return -3;
#endif
}

int mpcb_plant_step(mpcb_handle_t h, double* x, const double* u, const double* t, const double* pxp,
                    const double* pxmp, void* stream) {
#if !MPCB_PLANT_NOMINAL
    h->kernel_launches[KC_OTHER] += 1; h->host_launches += 1;
    k_plant_step<<<nblk(h->B, 128), 128, 0, (cudaStream_t)stream>>>(h->B, x, u, t, pxp, pxmp);
    CK(cudaGetLastError());
    return 0;
#else
    h->err = "nominal plant: use mpcb_model_step (MPC_code.py:813-814)"; return -3;
#endif
}

int mpcb_set_profiling(mpcb_handle_t h, int on) {
    h->profile = on ? 1 : 0;
    // events are created here, not inside a timed region (cudaEventCreate occasionally takes milliseconds when the
    // driver grows its pool: seen as 20-100 ms outliers on the steps that set a new record of launches)
    if (on) while (h->ev_pool.size() < 2 * 1024) { cudaEvent_t e; if (cudaEventCreate(&e) != cudaSuccess) break; h->ev_pool.push_back(e); }
    for (int i = 0; i < MPCB_NKERNELS; ++i) { h->kernel_ms[i] = 0.0; h->kernel_launches[i] = 0; }
    h->eval_instances = h->trial_instances = 0;
    CK(cudaDeviceSynchronize());
    CK(cudaMemset(h->counters, 0, 2 * sizeof(unsigned long long)));
    for (StepGroup* g : h->groups) {
        mpcb_ctx* c = g->c;
        c->profile = h->profile;
        for (int i = 0; i < MPCB_NKERNELS; ++i) { c->kernel_ms[i] = 0.0; c->kernel_launches[i] = 0; }
        c->eval_instances = c->trial_instances = 0;
        CK(cudaMemset(c->counters, 0, 2 * sizeof(unsigned long long)));
        if (on) while (c->ev_pool.size() < 2 * 1024) { cudaEvent_t e; if (cudaEventCreate(&e) != cudaSuccess) break; c->ev_pool.push_back(e); }
    }
    return 0;
}

int mpcb_get_profile(mpcb_handle_t h, double* kernel_ms, long* kernel_launches, unsigned long long* instance_counts) {
    for (int i = 0; i < MPCB_NKERNELS; ++i) { kernel_ms[i] = h->kernel_ms[i]; kernel_launches[i] = h->kernel_launches[i]; }
    instance_counts[0] = h->eval_instances; instance_counts[1] = h->trial_instances;
    for (StepGroup* g : h->groups) {        // grouped steps: sums over the groups (their kernels overlap in time)
        for (int i = 0; i < MPCB_NKERNELS; ++i) { kernel_ms[i] += g->c->kernel_ms[i]; kernel_launches[i] += g->c->kernel_launches[i]; }
        instance_counts[0] += g->c->eval_instances; instance_counts[1] += g->c->trial_instances;
    }
    return 0;
}

int mpcb_dfma_peak(int iters, double* tflops) {
    const int blocks = 148 * 16, threads = 256;
    double* out = nullptr;
    if (cudaMalloc(&out, sizeof(double) * blocks * threads) != cudaSuccess) return -1;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    k_dfma_peak<<<blocks, threads>>>(out, 1000);
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        k_dfma_peak<<<blocks, threads>>>(out, iters);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) { cudaFree(out); return -1; }
        float ms = 0.f; cudaEventElapsedTime(&ms, e0, e1);
        const double fl = 2.0 * 8.0 * (double)iters * blocks * threads;
        if (ms > 0.f && fl / (ms * 1e-3) / 1e12 > best) best = fl / (ms * 1e-3) / 1e12;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    *tflops = best;
    return 0;
}

int mpcb_loop_reset(mpcb_handle_t h, const double* x0_m, const double* u0, const double* dhat0, const double* P0) {
#if MPCB_HAS_OCP && MPCB_HAS_TARGET
    const size_t B = (size_t)h->B;
    if (!h->loop_mem) {
        const size_t n = B * (NXI + NXI * NXI + 3 * NU + 2 * NX + 3 * NW + MPCB_NPARSS + NWS + NPAR + NPX + NPY + 1);
        CK(cudaMalloc(&h->loop_mem, sizeof(double) * n));
        CK(cudaMalloc(&h->loop_imem, sizeof(int) * 3 * B));
        double* p = h->loop_mem;
        LoopState& L = h->L;
        L.xi = p; p += B * NXI; L.P = p; p += B * NXI * NXI; L.u = p; p += B * NU; L.us = p; p += B * NU; L.u0 = p; p += B * NU;
        L.xs = p; p += B * NX; L.x0m = p; p += B * NX; L.wguess = p; p += B * NW; L.wopt = p; p += B * NW; L.w = p; p += B * NW;
        L.parss = p; p += B * MPCB_NPARSS; L.wss = p; p += B * NWS; L.par = p; p += B * NPAR; L.px0 = p; p += B * NPX;
        L.py0 = p; p += B * NPY; L.fss = p; p += B;
        L.dyn_status = h->loop_imem; L.ss_status = h->loop_imem + B; L.ss_iters = h->loop_imem + 2 * B;
    }
    LoopState& L = h->L;
    CK(cudaMemset(h->loop_mem, 0, sizeof(double) * B * (NXI + NXI * NXI)));
    CK(cudaMemset(h->loop_imem, 0, sizeof(int) * 3 * B));
    CK(cudaMemcpy2D(L.xi, sizeof(double) * NXI, x0_m, sizeof(double) * NX, sizeof(double) * NX, B, cudaMemcpyDeviceToDevice));
    if (NXI > NX && dhat0)
        CK(cudaMemcpy2D(L.xi + NX, sizeof(double) * NXI, dhat0, sizeof(double) * ND, sizeof(double) * ND, B, cudaMemcpyDeviceToDevice));
    if (P0) CK(cudaMemcpy(L.P, P0, sizeof(double) * B * NXI * NXI, cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy(L.x0m, x0_m, sizeof(double) * B * NX, cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy(L.xs, x0_m, sizeof(double) * B * NX, cudaMemcpyDeviceToDevice));            // MPC_code.py:682-684
    CK(cudaMemcpy(L.u0, u0, sizeof(double) * B * NU, cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy(L.u, u0, sizeof(double) * B * NU, cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy(L.us, u0, sizeof(double) * B * NU, cudaMemcpyDeviceToDevice));
    h->loop_first = 1;
    return 0;
#else
    h->err = "library built without OCP/target"; return -3;
#endif
}

int mpcb_loop_get(mpcb_handle_t h, double* xi, double* P, double* u, void* stream) {
#if MPCB_HAS_OCP && MPCB_HAS_TARGET
    if (!h->loop_mem) { h->err = "mpcb_loop_reset has not been called"; return -2; }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t B = (size_t)h->B;
    if (xi) CK(cudaMemcpyAsync(xi, h->L.xi, sizeof(double) * B * NXI, cudaMemcpyDeviceToDevice, s));
    if (P) CK(cudaMemcpyAsync(P, h->L.P, sizeof(double) * B * NXI * NXI, cudaMemcpyDeviceToDevice, s));
    if (u) CK(cudaMemcpyAsync(u, h->L.u, sizeof(double) * B * NU, cudaMemcpyDeviceToDevice, s));
    return 0;
#else
    h->err = "library built without OCP/target"; return -3;
#endif
}

static int step_impl(mpcb_ctx* h, int est_type, const double* y_meas, const double* t, const double* sp, const double* px,
              const double* py, double* u_out, double* xhat_out, double* dhat_out, double* xs_out, double* us_out,
              double* f_dyn, int* status_dyn, int* iters_dyn, int* status_ss, void* stream) {
#if MPCB_HAS_OCP && MPCB_HAS_TARGET
    if (!h->loop_mem) { h->err = "mpcb_loop_reset has not been called"; return -2; }
    cudaStream_t s = (cudaStream_t)stream;
    LoopState& L = h->L;
    const int B = h->B, g = nblk(B, 128);
    k_step_params<<<g, 128, 0, s>>>(B, px, py, L);
    int rc = mpcb_estimate(h, est_type, y_meas, L.u, t, L.px0, L.py0, L.xi, L.P, s);
    if (rc) return rc;
    k_step_pre<<<g, 128, 0, s>>>(B, t, sp, L, xhat_out, dhat_out);
    rc = mpcb_target(h, L.parss, L.wss, L.fss, L.ss_status, L.ss_iters, s);
    if (rc) return rc;
    k_step_mid<<<nblk((long)B * 32, 128), 128, 0, s>>>(B, h->loop_first, t, px, py, L, xs_out, us_out);
    rc = mpcb_ocp(h, L.par, L.w, f_dyn, status_dyn, iters_dyn, s);
    if (rc) return rc;
    k_step_post<<<nblk((long)B * 32, 128), 128, 0, s>>>(B, t, status_dyn, L, u_out, h->hold_failed);
    if (status_ss) CK(cudaMemcpyAsync(status_ss, L.ss_status, sizeof(int) * B, cudaMemcpyDeviceToDevice, s));
    CK(cudaGetLastError());
    h->kernel_launches[KC_OTHER] += 4; h->host_launches += 4;
    h->loop_first = 0;
    return 0;
#else
    h->err = "library built without OCP/target"; return -3;
#endif
}


// ---------------------------------------------------------------------------------------------
// Instance groups.  The solve alternates throughput-bound kernels (stage derivatives) with latency-bound ones (the
// N-sequential Riccati sweep, the target solve, the tail of ticks in which only a few instances still iterate).
// Instances are independent, so the batch can be cut into G contiguous groups, each queued on its own stream: one group's
// latency-bound phase overlaps another's evaluation.  Every group's step is a handful of launches plus one CUDA-graph
// launch, all issued by the calling thread - no worker threads, nobody waits (round 1 needed one polling host thread per
// group, which made the number of groups a function of the host's core count).  Results are bit-identical to the
// ungrouped step.  Children alias the parent's buffers at an instance offset.
// ---------------------------------------------------------------------------------------------
#if MPCB_HAS_OCP && MPCB_HAS_TARGET
static int groups_setup(mpcb_ctx* h) {
    groups_teardown(h);
    const int G = h->ngroups, B = h->B, per = (B + G - 1) / G;
    if (!h->ev_in) CK(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
    for (int b0 = 0; b0 < B; b0 += per) {
        StepGroup* g = new StepGroup();
        g->b0 = b0; g->nb = (b0 + per <= B) ? per : B - b0;
        mpcb_ctx* c = new mpcb_ctx();
        // constants (bounds, filter matrices) are shared with the parent; everything a solve writes is the group's own
        c->device = h->device; c->opts_ss = h->opts_ss; c->opts_dyn = h->opts_dyn; c->have_dbounds = h->have_dbounds;
        c->lbx = h->lbx; c->ubx = h->ubx; c->lbg = h->lbg; c->ubg = h->ubg; c->ss_lbx = h->ss_lbx; c->ss_ubx = h->ss_ubx;
        c->Qkf = h->Qkf; c->Rkf = h->Rkf; c->Kest = h->Kest; c->dmin = h->dmin; c->dmax = h->dmax;
        c->loop_mem = h->loop_mem; c->loop_imem = h->loop_imem; c->loop_first = h->loop_first;
        c->profile = h->profile; c->host_loop = h->host_loop; c->ngroups = 1; c->ev_in = nullptr; c->hold_failed = h->hold_failed;
        c->og_graph = nullptr; c->og_exec = nullptr; c->og_valid = 0; c->host_launches = 0; c->last_stream = nullptr;
        c->eval_instances = c->trial_instances = 0;
        for (int i = 0; i < MPCB_NKERNELS; ++i) { c->kernel_ms[i] = 0.0; c->kernel_launches[i] = 0; }
        c->B = g->nb;
        c->ws = h->ws + (size_t)b0 * OcpLayout::total; c->st = h->st + b0;
        if (cudaMalloc(&c->n_active, sizeof(int)) != cudaSuccess || cudaMallocHost(&c->h_active, sizeof(int)) != cudaSuccess ||
            cudaMalloc(&c->counters, 2 * sizeof(unsigned long long)) != cudaSuccess ||
            cudaMalloc(&c->tick_ctr, 2 * sizeof(unsigned long long)) != cudaSuccess) { h->err = "group allocation failed"; return -1; }
        cudaMemset(c->counters, 0, 2 * sizeof(unsigned long long));
        cudaMemset(c->tick_ctr, 0, 2 * sizeof(unsigned long long));
        cudaMemset(c->n_active, 0, sizeof(int));
        const size_t o = (size_t)b0;
        LoopState& L = c->L; const LoopState& P = h->L;
        L.xi = P.xi + o * NXI; L.P = P.P + o * NXI * NXI; L.u = P.u + o * NU; L.us = P.us + o * NU; L.u0 = P.u0 + o * NU;
        L.xs = P.xs + o * NX; L.x0m = P.x0m + o * NX; L.wguess = P.wguess + o * NW; L.wopt = P.wopt + o * NW; L.w = P.w + o * NW;
        L.parss = P.parss + o * MPCB_NPARSS; L.wss = P.wss + o * NWS; L.par = P.par + o * NPAR; L.px0 = P.px0 + o * NPX;
        L.py0 = P.py0 + o * NPY; L.fss = P.fss + o;
        L.dyn_status = P.dyn_status + o; L.ss_status = P.ss_status + o; L.ss_iters = P.ss_iters + o;
        g->c = c;
        if (cudaStreamCreateWithFlags(&g->s, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&g->done, cudaEventDisableTiming) != cudaSuccess) { h->err = "group stream creation failed"; return -1; }
        h->groups.push_back(g);
    }
    return 0;
}
#endif

static void groups_teardown(mpcb_ctx* h) {
#if MPCB_HAS_OCP && MPCB_HAS_TARGET
    for (StepGroup* g : h->groups) {
        cudaStreamSynchronize(g->s);
        h->host_launches += g->c->host_launches;              // keep the totals of mpcb_total_launches monotone
        unsigned long long ctr[2] = {0, 0};
        cudaMemcpy(ctr, g->c->tick_ctr, sizeof(ctr), cudaMemcpyDeviceToHost);
        h->host_launches += TICK_KERNELS * (long)ctr[1];
        cudaStreamDestroy(g->s); cudaEventDestroy(g->done);
        ocp_graph_drop(g->c);
        cudaFree(g->c->n_active); cudaFreeHost(g->c->h_active); cudaFree(g->c->counters); cudaFree(g->c->tick_ctr);
        for (auto e : g->c->ev_pool) cudaEventDestroy(e);
        delete g->c; delete g;
    }
#endif
    h->groups.clear();
}

int mpcb_set_policy(mpcb_handle_t h, int hold_failed) { h->hold_failed = hold_failed ? 1 : 0; return 0; }

int mpcb_set_groups(mpcb_handle_t h, int n) {
    if (n < 1 || n > h->B) { h->err = "mpcb_set_groups: need 1 <= n <= batch"; return -2; }
    if (n != h->ngroups) { groups_teardown(h); h->ngroups = n; }
    return 0;
}

// Asynchronous: every launch of the step is queued behind the caller's work on `stream`, and `stream` is made to wait for
// the step's completion; the call returns without waiting.  Read the outputs in stream order (or after synchronising).
int mpcb_step(mpcb_handle_t h, int est_type, const double* y_meas, const double* t, const double* sp, const double* px,
              const double* py, double* u_out, double* xhat_out, double* dhat_out, double* xs_out, double* us_out,
              double* f_dyn, int* status_dyn, int* iters_dyn, int* status_ss, void* stream) {
#if MPCB_HAS_OCP && MPCB_HAS_TARGET
    h->last_stream = (cudaStream_t)stream;
    if (h->ngroups <= 1)
        return step_impl(h, est_type, y_meas, t, sp, px, py, u_out, xhat_out, dhat_out, xs_out, us_out, f_dyn, status_dyn,
                         iters_dyn, status_ss, stream);
    if (!h->loop_mem) { h->err = "mpcb_loop_reset has not been called"; return -2; }
    if (h->groups.empty()) { int rc = groups_setup(h); if (rc) return rc; }
    CK(cudaEventRecord(h->ev_in, (cudaStream_t)stream));      // the groups start after the caller's work on `stream`
    int rc = 0;
    for (StepGroup* g : h->groups) {
        const size_t o = (size_t)g->b0;
        mpcb_ctx* c = g->c;
        c->opts_ss = h->opts_ss; c->opts_dyn = h->opts_dyn; c->have_dbounds = h->have_dbounds; c->loop_first = h->loop_first;
        c->profile = h->profile; c->hold_failed = h->hold_failed;
        CK(cudaStreamWaitEvent(g->s, h->ev_in, 0));
        const int r = step_impl(c, est_type, y_meas + o * NY, t + o, sp + o * (NU + NY + NX), px ? px + o * NPX * NH : nullptr,
                                py ? py + o * NPY * NH : nullptr, u_out + o * NU, xhat_out + o * NX, dhat_out + o * ND,
                                xs_out + o * NX, us_out + o * NU, f_dyn + o, status_dyn + o, iters_dyn + o,
                                status_ss ? status_ss + o : nullptr, g->s);
        if (r && !rc) { rc = r; h->err = c->err; }
        CK(cudaEventRecord(g->done, g->s));
        CK(cudaStreamWaitEvent((cudaStream_t)stream, g->done, 0));
    }
    h->loop_first = 0;
    return rc;
#else
    h->err = "library built without OCP/target"; return -3;
#endif
}

// Counters.  The device-driven solve counts its ticks on the device, so these wait for the handle's last stream first.
static void read_ticks(mpcb_ctx* h, unsigned long long* last, unsigned long long* total) {
    unsigned long long ctr[2] = {0, 0};
    cudaStreamSynchronize(h->last_stream);
    cudaMemcpy(ctr, h->tick_ctr, sizeof(ctr), cudaMemcpyDeviceToHost);
    *last = ctr[0]; *total = ctr[1];
}

int mpcb_last_ticks(mpcb_handle_t h) {
    if (h->last_ticks >= 0 && h->groups.empty()) return h->last_ticks;       // host-polled solve: counted on the host
    unsigned long long last = 0, total = 0, worst = 0;
    if (h->groups.empty()) { read_ticks(h, &last, &total); return (int)last; }
    for (StepGroup* g : h->groups) {
        cudaStreamSynchronize(g->s);
        if (g->c->last_ticks >= 0) { worst = worst > (unsigned long long)g->c->last_ticks ? worst : (unsigned long long)g->c->last_ticks; continue; }
        read_ticks(g->c, &last, &total);
        worst = worst > last ? worst : last;
    }
    return (int)worst;
}

// kernel launches made through this handle since its creation (host launches + TICK_KERNELS per device-driven tick)
long mpcb_total_launches(mpcb_handle_t h) {
    unsigned long long last = 0, total = 0;
    read_ticks(h, &last, &total);
    long n = h->host_launches + TICK_KERNELS * (long)total;
    for (StepGroup* g : h->groups) {
        cudaStreamSynchronize(g->s);
        read_ticks(g->c, &last, &total);
        n += g->c->host_launches + TICK_KERNELS * (long)total;
    }
    return n;
}

int mpcb_last_launches(mpcb_handle_t h) { return h->last_launches; }

}  // extern "C"
