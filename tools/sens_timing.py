"""Cost of the OCP sensitivities on the GPU, against the solve they belong to (Ex_NMPC, B = 4096 by default).

CUDA events around, after warm-up: the batched mpcb_ocp solve, mpcb_ocp_sens_factor, the full theta-Jacobian (one JVP
of all ntheta unit directions) and one VJP; for p = [d | px | py] mpcb_ocp_sens_factor_p, the d-Jacobian (nd unit
directions), the full p-Jacobian (all n_p unit directions) and one VJP_p; for the target problem the batched mpcb_target
solve, mpcb_target_sens_factor (which solves again), the full theta_ss-Jacobian and one VJP; the median of --reps
repetitions each.  Prints the card name and power limit read in the same run.  Usage: python tools/sens_timing.py [--batch 4096] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as entry
    from mpc_code_b200.mpc_loop import CompiledProblem
    from mpc_code_b200.solvers import BatchedNlpSolver, MpcbHandle
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    prob, ss, ocp = entry._problem("nmpc_cstr")
    cp = CompiledProblem(prob, "nmpc_cstr")
    G = np.load(os.path.join(ROOT, "tests", "golden", "nmpc_oracle.npz"))
    B = a.batch
    rng = np.random.default_rng(0)
    par = G["ocp_par"][np.arange(B) % G["ocp_par"].shape[0]].copy()
    par[:, :2 * prob.nx] *= 1 + 0.002 * rng.uniform(-1, 1, (B, 2 * prob.nx))
    h = MpcbHandle(cp.library, B)
    solver = BatchedNlpSolver("ocp", cp.ocp_spec).attach(h)
    par_t = h.tensor(par, prob.npar)
    w0 = h.tensor(G["ocp_w0"], prob.nw)
    nth = h.ntheta
    eye = torch.eye(nth, dtype=torch.float64, device=h.device).expand(B, -1, -1).contiguous()
    gw = torch.as_tensor(rng.standard_normal((B, prob.nw)), device=h.device)

    def timed(fn):
        out = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return float(np.median(out))

    solver(x0=w0, p=par_t)                                   # warm-up: graph build, module load
    sens = solver.sensitivity(); sens.jvp(eye); sens.vjp(gw); torch.cuda.synchronize()
    t_solve = timed(lambda: solver(x0=w0, p=par_t))
    solver(x0=w0, p=par_t)
    t_factor = timed(lambda: h.ocp_sens_factor(par_t))
    fac, st = h.ocp_sens_factor(par_t)
    t_jac = timed(lambda: h.ocp_jvp(fac, eye))
    t_vjp = timed(lambda: h.ocp_vjp(fac, gw))
    npp = h.np_params
    eye_p = torch.eye(npp, dtype=torch.float64, device=h.device).expand(B, -1, -1).contiguous()
    eye_d = eye_p[:, :prob.nd].contiguous()
    t_factor_p = timed(lambda: h.ocp_sens_factor_p(par_t))
    fac_p, st_p = h.ocp_sens_factor_p(par_t)
    h.ocp_jvp_p(fac_p, eye_p); h.ocp_vjp_p(fac_p, gw); torch.cuda.synchronize()
    t_jac_d = timed(lambda: h.ocp_jvp_p(fac_p, eye_d))
    t_jac_p = timed(lambda: h.ocp_jvp_p(fac_p, eye_p))
    t_vjp_p = timed(lambda: h.ocp_vjp_p(fac_p, gw))
    # target problem: the golden instances with perturbed disturbance estimates and output set-points
    par_ss = G["ss_par"][np.arange(B) % G["ss_par"].shape[0]].copy()
    o = ss.off
    par_ss[:, o["ysp"]:o["xsp"]] *= 1 + 0.01 * rng.uniform(-1, 1, (B, prob.ny))
    par_ss[:, o["d"]:o["usprev"]] *= 1 + 0.01 * rng.uniform(-1, 1, (B, prob.nd))
    par_ss = h.tensor(par_ss, ss.npar)
    wss0 = h.tensor(G["ss_w0"][np.arange(B) % G["ss_w0"].shape[0]], ss.nw)
    solver_ss = BatchedNlpSolver("target", ss).attach(h)
    eye_ss = torch.eye(h.ntheta_ss, dtype=torch.float64, device=h.device).expand(B, -1, -1).contiguous()
    gws = torch.as_tensor(rng.standard_normal((B, ss.nw)), device=h.device)
    solver_ss(x0=wss0, p=par_ss)
    fac_t, st_t = h.target_sens_factor(par_ss, wss0)
    h.target_jvp(fac_t, eye_ss); h.target_vjp(fac_t, gws); torch.cuda.synchronize()
    t_tsolve = timed(lambda: h.target(par_ss, wss0))
    t_tfactor = timed(lambda: h.target_sens_factor(par_ss, wss0))
    t_tjac = timed(lambda: h.target_jvp(fac_t, eye_ss))
    t_tvjp = timed(lambda: h.target_vjp(fac_t, gws))
    res = dict(card=card, problem="nmpc_cstr (Ex_NMPC)", batch=B, ntheta=nth, reps=a.reps,
               sens_status_counts={int(k): int(v) for k, v in zip(*np.unique(st.cpu().numpy(), return_counts=True))},
               solve_ms=t_solve, factor_ms=t_factor, jacobian_ms=t_jac, vjp_ms=t_vjp,
               factor_plus_jacobian_over_solve=(t_factor + t_jac) / t_solve, vjp_over_solve=t_vjp / t_solve,
               factor_plus_vjp_over_solve=(t_factor + t_vjp) / t_solve,
               n_p=npp, capture_p_doubles_per_instance=int(h.L.mpcb_ocp_sens_size_p()),
               sens_p_status_counts={int(k): int(v) for k, v in zip(*np.unique(st_p.cpu().numpy(), return_counts=True))},
               factor_p_ms=t_factor_p, d_jacobian_ms=t_jac_d, p_jacobian_ms=t_jac_p, vjp_p_ms=t_vjp_p,
               factor_p_plus_d_jacobian_over_solve=(t_factor_p + t_jac_d) / t_solve,
               factor_p_plus_p_jacobian_over_solve=(t_factor_p + t_jac_p) / t_solve,
               factor_p_plus_vjp_p_over_solve=(t_factor_p + t_vjp_p) / t_solve,
               ntheta_ss=h.ntheta_ss, capture_target_doubles_per_instance=int(h.L.mpcb_target_sens_size()),
               target_sens_status_counts={int(k): int(v) for k, v in zip(*np.unique(st_t.cpu().numpy(), return_counts=True))},
               target_solve_ms=t_tsolve, target_factor_ms=t_tfactor, target_jacobian_ms=t_tjac, target_vjp_ms=t_tvjp,
               target_factor_over_target_solve=t_tfactor / t_tsolve,
               target_factor_plus_jacobian_over_ocp_solve=(t_tfactor + t_tjac) / t_solve)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
