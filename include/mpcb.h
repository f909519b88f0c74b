/*
 * mpcb.h - C ABI of the batched MPC step solver (one shared library per compiled problem).
 *
 * The reference (CPCLAB-UNIPI/MPC-code) has no FFI: its loop is written against CasADi objects.
 * Each entry point below replaces one of those call sites for a whole batch of independent
 * instances; the reference site it stands in for is cited.  The Python host in
 * mpc-code_b200/ binds these with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *  - every data pointer is DEVICE memory (float64 / int32), instance-major: element j of
 *    instance i lives at ptr[i * len + j]; the caller owns all buffers;
 *  - `stream` is a cudaStream_t passed as void*; kernels are enqueued on it and EVERY call is asynchronous: outputs
 *    are complete when the stream reaches that point.  The iterative solves (mpcb_ocp, mpcb_step) are device driven -
 *    one CUDA graph whose WHILE node repeats the solver tick until no instance iterates - so the host never waits on
 *    them.  (With profiling on, see mpcb_set_profiling, they run a host-polled schedule and return when done.);
 *  - return value 0 = OK, < 0 = error (text via mpcb_last_error); a handle is bound to the
 *    device that was current at mpcb_create and is not thread-safe;
 *  - problem sizes and the user's model are compiled in (generated header); mpcb_get_dims
 *    reports them so the host can check its buffers.
 *  - per-instance solver status uses IPOPT's ApplicationReturnStatus values so that the host
 *    can answer solver.stats()['return_status'] like the reference's loop expects
 *    (MPC_code.py:714,786): 0 Solve_Succeeded, 1 Solved_To_Acceptable_Level,
 *    2 Infeasible_Problem_Detected, -1 Maximum_Iterations_Exceeded, -2 Restoration_Failed,
 *    -3 Error_In_Step_Computation, -13 Invalid_Number_Detected.
 */
#ifndef MPCB_H
#define MPCB_H

#ifdef __cplusplus
extern "C" {
#endif

#define MPCB_ABI_VERSION 2

typedef struct mpcb_ctx* mpcb_handle_t;

typedef struct mpcb_dims {
    int nx, nu, ny, nd, npx, npy;      /* MPC_code.py:31-48 */
    int nxp, npxp, npyp;               /* plant sizes */
    int nxi;                           /* estimator state size: nx (+ nd when offree != 'no') */
    int N, Mx;                         /* horizon, RK4 sub-steps per interval */
    int nw, npar, ng;                  /* OCP: variables, parameters (Control_Calc.py:31-57), range rows per stage */
    int nwss, nparss;                  /* target problem sizes (Target_Calc.py:29,41) */
    int has_ocp, has_target;
} mpcb_dims_t;

/* Interior-point options; names and defaults are IPOPT's (the reference sets only max_iter and
 * hessian_constant, MPC_code.py:262-263). */
typedef struct mpcb_opts {
    int    max_iter;                   /* Sol_itmax: 100 (Default_Values.py:102) */
    double tol;                        /* 1e-8 */
    double mu_init;                    /* 0.1 */
    double bound_relax_factor;         /* 1e-8 */
    int    honor_original_bounds;      /* 0 (IPOPT >= 3.14), 1 (IPOPT 3.12) */
    double bound_push;                 /* 1e-2 (also bound_frac) */
    double acceptable_tol;             /* 1e-6 */
    int    acceptable_iter;            /* 15 */
} mpcb_opts_t;

int  mpcb_abi_version(void);
void mpcb_default_opts(mpcb_opts_t* opts);
int  mpcb_get_dims(mpcb_dims_t* dims);

/* Algorithmic operation counts of the generated model functions (name -> flops), for roofline
 * accounting; returns the count for `name`, or -1 when unknown. */
long mpcb_model_flops(const char* name);

int  mpcb_create(int batch, const mpcb_opts_t* opts_ss, const mpcb_opts_t* opts_dyn, mpcb_handle_t* out);
int  mpcb_destroy(mpcb_handle_t h);
const char* mpcb_last_error(mpcb_handle_t h);

/* Shared (not per-instance) constants, copied from HOST memory:
 *   "ocp_lbx","ocp_ubx" [nw]  - w_lb / w_ub of opt_dyn (Control_Calc.py:213-252); entries 0..nx-1
 *                               are ignored, x0 is fixed from par[0:nx] (MPC_code.py:734)
 *   "ocp_lbg","ocp_ubg" [ng*N]- the range rows of g_lb / g_ub, stage by stage: for k = 0..N-1 the ny bounds of
 *                               Y_k (Control_Calc.py:227-230), the nu bounds of DU_k (:241-243) and the bounds
 *                               (-inf, 0) of the user inequalities G_k (:244-245); ng counts the blocks that are present
 *   "ss_lbx","ss_ubx"   [nwss]- wss_lb / wss_ub of opt_ss (Target_Calc.py:127-134)
 *   "Q_kf" [nxi*nxi], "R_kf" [ny*ny], "K_est" [nxi*ny] (row-major), "dmin","dmax" [nd]
 */
int  mpcb_set_const(mpcb_handle_t h, const char* name, const double* host_ptr, int n);

/* Estimator update (MPC_code.py:546-668 -> Estimator.py:231-386).
 * est_type 0: xi = xi- + K (y - Fy(xi-))           (kalss / Luenberger, Estimator.py:253-259)
 * est_type 1: Kalman / extended Kalman filter        (Estimator.py:263-311, 313-386)
 * xi [B,nxi] and P [B,nxi*nxi] (row-major) are updated in place; afterwards the d-part of xi is
 * clipped to [dmin,dmax] when those constants were set (MPC_code.py:659-665). */
int  mpcb_estimate(mpcb_handle_t h, int est_type, const double* y_meas, const double* u_prev, const double* t,
                   const double* px, const double* py, double* xi, double* P, void* stream);

/* Target problem solve (MPC_code.py:704-709 -> Target_Calc.py:20-161).
 * par_ss [B,nparss]; wss [B,nwss] initial guess in, solution out; fss [B]; status, iters [B]. */
int  mpcb_target(mpcb_handle_t h, const double* par_ss, double* wss, double* fss, int* status, int* iters,
                 void* stream);

/* Dynamic OCP solve (MPC_code.py:776-781 -> Control_Calc.py:20-260).
 * par [B,npar]; w [B,nw] initial guess in, solution out; f [B]; status, iters [B]. */
int  mpcb_ocp(mpcb_handle_t h, const double* par, double* w, double* f, int* status, int* iters, void* stream);

/* Sensitivities of the OCP solution with respect to theta = [x_hat (nx) | x_s (nx) | u_s (nu) | u_{k-1} (nu)]
 * (par[0 : 2nx+nu] and par[2nx+nu+nd : 2nx+2nu+nd]; ntheta = 2 (nx+nu)).  At the returned iterate of an instance the
 * primal-dual barrier system F(v; theta) = 0 that the solver iterates on is differentiated (implicit function
 * theorem, as sIPOPT does): bound multipliers and range-row slacks are condensed as in the Newton step (Sigma = Z/D,
 * no regularisation) and x_0 is eliminated, so dw[0:nx] = dx_hat exactly.  Strongly active bounds therefore give
 * derivatives of the order of the final barrier parameter, inactive ones the unconstrained derivative.  The
 * parameters d, t, lambda, px, py are held constant.
 *   mpcb_ocp_sens_size:   doubles per instance of the capture buffer `fac`.
 *   mpcb_ocp_sens_factor: after mpcb_ocp on the same handle and with that call's par; factors the solution's KKT
 *                         matrix (one Riccati sweep with delta_w = 0) and writes everything the sweeps need into
 *                         fac [B, size].  status [B]: 0 computed; 1 the solve's status was not 0 or 1; 2 wrong inertia
 *                         (some R~_k not positive definite, or a singular terminal-equality Gramian).  Any status
 *                         other than 0 makes that instance's outputs of the sweeps NaN.  The solver's workspace is
 *                         only read.
 *   mpcb_ocp_jvp:         dw [B, ndir, nw] = J dtheta for dtheta [B, ndir, ntheta], J = d(w opt)/d(theta), in the
 *                         caller's w layout.
 *   mpcb_ocp_vjp:         gtheta [B, ntheta] = J' gw for gw [B, nw].
 * The sweeps read only fac: their results do not depend on what the handle did after the factor call.  A problem
 * whose ContForm cost integrand depends on theta cannot provide these derivatives: jvp / vjp return < 0. */
long mpcb_ocp_sens_size(void);
int  mpcb_ocp_sens_factor(mpcb_handle_t h, const double* par, double* fac, int* status, void* stream);
int  mpcb_ocp_jvp(mpcb_handle_t h, const double* fac, int ndir, const double* dtheta, double* dw, void* stream);
int  mpcb_ocp_vjp(mpcb_handle_t h, const double* fac, const double* gw, double* gtheta, void* stream);

/* Sensitivities of the OCP solution with respect to the parameters that enter the dynamics,
 *   p = [d (nd) | px_0 .. px_{N-1} (npx N) | py_0 .. py_{N-1} (npy N)] = par[2nx+nu : 2nx+nu+nd] ++ par[off_px : npar]
 * (n_p = nd + (npx+npy) N; off_px = 2nx+2nu+nd+1+ny*nu).  The same derivative as above (theta held constant, t and
 * lambda too); p enters the model's state map, so the sweeps carry the defects (dF_k/dp_k) dp_k of the dynamics rows.
 *   mpcb_ocp_sens_size_p:   doubles per instance of the capture of mpcb_ocp_sens_factor_p.
 *   mpcb_ocp_sens_factor_p: as mpcb_ocp_sens_factor (same status), into fac [B * size_p]: the first B * size doubles
 *                           are exactly what mpcb_ocp_sens_factor writes, so the theta entry points accept this
 *                           capture; the derivative blocks of p follow.  Element 1 of an instance's theta capture
 *                           is set to 1 to mark that its p-blocks are present.
 *   mpcb_ocp_jvp_p:         dw [B, ndir, nw] = J_p dp for dp [B, ndir, n_p].
 *   mpcb_ocp_vjp_p:         gp [B, n_p] = J_p' gw for gw [B, nw].
 * The p sweeps write NaN for an instance whose status is not 0 and for one whose capture has no p-blocks (element 1
 * of its theta capture is not 1, e.g. a zero-filled buffer of size_p that only mpcb_ocp_sens_factor wrote).
 * mpcb_ocp_sens_factor does not clear that mark: refresh a p capture with mpcb_ocp_sens_factor_p.  A ContForm problem,
 * a large model on the dense derivative path (MPCB_DENSE_SH) or a stage map that reads another stage's px / py through
 * par cannot provide the p-blocks (decided at code generation): the three p entry points return < 0. */
long mpcb_ocp_sens_size_p(void);
int  mpcb_ocp_sens_factor_p(mpcb_handle_t h, const double* par, double* fac, int* status, void* stream);
int  mpcb_ocp_jvp_p(mpcb_handle_t h, const double* fac, int ndir, const double* dp, double* dw, void* stream);
int  mpcb_ocp_vjp_p(mpcb_handle_t h, const double* fac, const double* gw, double* gp, void* stream);

/* Sensitivities of the steady-state target solution with respect to
 *   theta_ss = [usp (nu) | ysp (ny) | xsp (nx) | d (nd) | Us_prev (nu) | px (npx) | py (npy)]
 * (par_ss without vec(lambda) and t, which are held constant; ntheta_ss = 2nu+ny+nx+nd+npx+npy).  The derivative of
 * the OCP's kind applied to the target's barrier KKT system at the returned iterate: K of the Newton step (Hessian of
 * the Lagrangian + Sigma = Z/D, with the slacks of User_g_ineq_SS condensed like any bounded variable) without
 * regularisation, dwss/dtheta_ss = -[K^-1 dF/dtheta_ss]_{0:nwss}.  With honor_original_bounds it is taken at the
 * iterate before the final clipping.  mpcb_target keeps no workspace, so the factor call solves the problem again,
 * from the same guess and with the same code, and captures at its end.
 *   mpcb_target_sens_size:   doubles per instance of the capture `fac`: [0] its status, [1] the solve's status,
 *                            [2 : 2+nwss] the solution, then the Bunch-Kaufman factor of K, its pivots, dF/dtheta_ss.
 *   mpcb_target_sens_factor: par_ss and wss0 as given to mpcb_target (wss0 is not modified; the stored wss equals that
 *                            call's output); writes only fac [B, size] and status [B]: 0 computed; 1 the solve's status
 *                            was not 0 or 1; 2 wrong inertia of K.  Any status other than 0 makes that instance's
 *                            outputs of jvp / vjp NaN.
 *   mpcb_target_jvp:         dwss [B, ndir, nwss] = T dth for dth [B, ndir, ntheta_ss], T = d(wss opt)/d(theta_ss).
 *   mpcb_target_vjp:         gth [B, ntheta_ss] = T' gwss for gwss [B, nwss].
 * Without the target problem, or for a large model on the dense derivative path (decided at code generation), all
 * four return < 0. */
long mpcb_target_sens_size(void);
int  mpcb_target_sens_factor(mpcb_handle_t h, const double* par_ss, const double* wss0, double* fac, int* status, void* stream);
int  mpcb_target_jvp(mpcb_handle_t h, const double* fac, int ndir, const double* dth, double* dwss, void* stream);
int  mpcb_target_vjp(mpcb_handle_t h, const double* fac, const double* gwss, double* gth, void* stream);

/* Plant measurement  y = Fy_p(x,u,pyp,t,pymp) + noise   (MPC_code.py:531-541); noise may be NULL. */
int  mpcb_plant_meas(mpcb_handle_t h, const double* x, const double* u, const double* t, const double* pyp,
                     const double* pymp, const double* noise, double* y, void* stream);

/* Plant step  x <- Fx_p(x,u,pxp,t,h,pxmp)   (MPC_code.py:813-816), in place. */
int  mpcb_plant_step(mpcb_handle_t h, double* x, const double* u, const double* t, const double* pxp,
                     const double* pxmp, void* stream);

/* Model maps used by the loop glue: y = Fy_model(x,u,d,t,py) (MPC_code.py:524,699,730) and
 * x+ = Fx_model(x,u,h,d,t,px) (MPC_code.py:805). */
int  mpcb_model_output(mpcb_handle_t h, const double* x, const double* u, const double* d, const double* t,
                       const double* py, double* y, void* stream);
int  mpcb_model_step(mpcb_handle_t h, const double* x, const double* u, const double* d, const double* t,
                     const double* px, double* xn, void* stream);

/* Stage derivative evaluation on its own (the dominant kernel, exposed for tests and profiling):
 * for every instance i and stage k computes, at w and multipliers lam [B,N*nx]:
 *   A [B,N,nx*nx], Bm [B,N,nx*nu] (column-major), c [B,N,nx] = Fx_model(x_k,u_k) - x_{k+1},
 *   H [B,N,nz(nz+1)/2] = packed lower triangle of the Hessian of lam_{k+1}' Fx_model wrt (x_k,u_k). */
int  mpcb_stage_derivs(mpcb_handle_t h, const double* par, const double* w, const double* lam,
                       double* A, double* Bm, double* c, double* H, void* stream);

/* Fused closed-loop step (the throughput entry point): estimator -> target -> OCP -> extraction with the loop state
 * (x_hat, d_hat, P, u_{k-1}, targets, warm start) kept on the device between calls, i.e. MPC_code.py:546-805 for
 * every instance without host glue.
 *   mpcb_loop_reset: initial loop state (MPC_code.py:442-463); x0_m [B,nx], u0 [B,nu], dhat0 [B,nd] or NULL, P0 [B,nxi*nxi] or NULL.
 *   mpcb_step: y_meas [B,ny] measurement; t [B]; sp [B, nu+ny+nx] = usp|ysp|xsp (defSP, MPC_code.py:679);
 *              px [B,npx*N], py [B,npy*N] horizon parameters (MPC_code.py:492-501) or NULL for zeros;
 *              outputs u_out [B,nu] (input to apply), xhat_out [B,nx] / dhat_out [B,nd] (x(k|k), d(k|k)),
 *              xs_out / us_out (targets), f_dyn, status_dyn, iters_dyn, status_ss [B].
 *   mpcb_loop_get: copies the kept state (xi = [x(k+1|k); d] [B,nxi], P [B,nxi*nxi], u [B,nu]; any may be NULL) out.
 */
int  mpcb_loop_reset(mpcb_handle_t h, const double* x0_m, const double* u0, const double* dhat0, const double* P0);
int  mpcb_step(mpcb_handle_t h, int est_type, const double* y_meas, const double* t, const double* sp, const double* px,
               const double* py, double* u_out, double* xhat_out, double* dhat_out, double* xs_out, double* us_out,
               double* f_dyn, int* status_dyn, int* iters_dyn, int* status_ss, void* stream);
int  mpcb_loop_get(mpcb_handle_t h, double* xi, double* P, double* u, void* stream);

/* Instance groups of the fused step: mpcb_step cuts the batch into n contiguous groups, each queued on its own CUDA
 * stream (all launches made by the calling thread), so that the latency-bound phases of one group (Riccati sweep,
 * target solve, the tail of iterations in which few instances are still active) overlap the evaluation kernels of
 * another.  Results do not change (instances are independent - the reference solves them one after another,
 * MPC_code.py:485).  The caller's stream is made to wait for all groups.  Default 1. */
int  mpcb_set_groups(mpcb_handle_t h, int n);

/* Policy of the fused step for FAILED solves (status < 0: Maximum_Iterations_Exceeded, Restoration_Failed,
 * Error_In_Step_Computation).  0 (default) = the reference's behaviour: only Infeasible_Problem_Detected is rejected, any
 * other iterate is applied to the plant (MPC_code.py:786).  1 = hold: treat them like an infeasible solve (previous input
 * kept, estimate propagated with the model, warm start kept; MPC_code.py:804-805). */
int  mpcb_set_policy(mpcb_handle_t h, int hold_failed);

/* Profiling.  With profiling on, every kernel launch is bracketed by CUDA events on its stream and the
 * time is accumulated per kernel class: 0 ocp_init, 1 ocp_eval (stage derivatives), 2 ocp_kkt (Riccati
 * step), 3 ocp_trial (line-search evaluation), 4 ocp_accept, 5 target, 6 estimate, 7 other.
 * instance_counts[0] = number of (instance) derivative evaluations done by class 1,
 * instance_counts[1] = number of (instance) trial evaluations done by class 3.
 * mpcb_set_profiling resets the accumulators.  Launch counts are kept even with profiling off. */
int  mpcb_set_profiling(mpcb_handle_t h, int on);
int  mpcb_get_profile(mpcb_handle_t h, double* kernel_ms /*[8]*/, long* kernel_launches /*[8]*/,
                      unsigned long long* instance_counts /*[2]*/);

/* FP64 FMA issue-rate micro-benchmark of the current device (8 independent chains per thread):
 * the measured denominator for FP64 roofline fractions (MEASURED_PEAKS.json has no FP64 entry). */
int  mpcb_dfma_peak(int iters, double* tflops);

/* Counters.  mpcb_last_ticks: solver ticks of the last OCP solve (largest over the groups); mpcb_total_launches:
 * kernel launches made through the handle since mpcb_create, the ticks of the device-driven solves included (4 launches
 * each).  Both wait for the handle's streams - the tick counts live on the device.  mpcb_last_launches: launches of the
 * last host-polled call, -1 after a device-driven one. */
int  mpcb_last_launches(mpcb_handle_t h);
int  mpcb_last_ticks(mpcb_handle_t h);
long mpcb_total_launches(mpcb_handle_t h);

#ifdef __cplusplus
}
#endif
#endif /* MPCB_H */
