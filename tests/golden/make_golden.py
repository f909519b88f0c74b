"""Regenerate the committed fixtures from an unmodified CPCLAB-UNIPI/MPC-code checkout:

    MPC_CODE_REFERENCE=<checkout> python tests/golden/make_golden.py

* ``kat.json``  - known-answer facts read from the reference's own example files (SURVEY.md section 4):
  KAT1 steady state of Ex_NMPC.py, KAT2 the printed linearisation in Ex_LMPC_nlplant.py:85-91,
  KAT3 closed-form targets derived from Ex_NMPC.py:129-148,217-219,241-242.
* ``ref_examples_oracle.npz`` - oracle closed loops of the unmodified Ex_NMPC_dis.py and Ex_LMPCxp_nlplant.py.
* ``nmpc_oracle.npz`` - outputs of the CPU oracle on the UNMODIFIED Ex_NMPC.py of the checkout
  (loaded through the casadi stand-in): OCP and target solutions, EKF updates, a short closed loop.
* ``problem_records.json`` - what defines each problem (tests/problem_record.py) of the unmodified files that
  examples/ restates (``--only-problem-records``).  ``--only-problem-records --from-examples`` records the
  restatements instead, for use where no checkout exists; the file names its source.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
import mpc_code_b200  # noqa: E402,F401
from mpc_code_b200.loader import load_example  # noqa: E402
from mpc_code_b200.problem import build_problem, make_specs  # noqa: E402
from oracle import cmodel, estimators  # noqa: E402
from oracle.closed_loop import OracleLoop  # noqa: E402
from oracle.ipm import IpmOptions  # noqa: E402
from oracle.nlp import OcpNlp, TargetNlp  # noqa: E402

REF = os.environ.get("MPC_CODE_REFERENCE", "")


def make_synthetic(names):
    """Oracle solutions of members of the synthetic family (symbolic Hessians of the unrolled RK4 graph take minutes to
    build for 8+ states - hence fixtures); members already in the file and not named are kept."""
    import __graft_entry__ as entry
    syn_path = os.path.join(HERE, "synthetic_oracle.npz")
    syn = dict(np.load(syn_path)) if os.path.exists(syn_path) else {}        # members not named are kept
    for name in names:
        p_s, ss_s, ocp_s = entry._problem(name)
        mod_s = cmodel.build(name, p_s, ocp_s, ss_s)
        on_s = OcpNlp(ocp_s, mod_s)
        rng_s = np.random.default_rng(5)
        nxs, nus, Ns_ = p_s.nx, p_s.nu, p_s.N
        nz_s = nxs + nus
        w0s = np.zeros(ocp_s.nw)
        pars, Ws, Fs, STs, ITs = [], [], [], [], []
        for _ in range(4):
            xh = rng_s.uniform(-1, 1, nxs)
            par_s = np.concatenate([xh, np.zeros(nxs), np.zeros(nus), np.zeros(0), np.zeros(nus), [0.0], np.zeros(p_s.ny * nus),
                                    np.zeros((p_s.npx + p_s.npy) * Ns_)])
            lb, ub = ocp_s.w_lb.copy(), ocp_s.w_ub.copy(); lb[:nxs] = ub[:nxs] = xh
            r = on_s.solve(w0s, par_s, lb, ub, opts=IpmOptions(max_iter=100))
            pars.append(par_s); Ws.append(r.x); Fs.append(r.f); STs.append(r.status); ITs.append(r.iters)
            print(name, r.return_status, r.iters, r.f)
        syn.update({name + "_par": np.array(pars), name + "_w": np.array(Ws), name + "_f": np.array(Fs),
                    name + "_status": np.array(STs), name + "_iters": np.array(ITs)})
    np.savez_compressed(syn_path, **syn)


def make_reference_examples():
    """Oracle closed loops of the UNMODIFIED reference files that the BASELINE configurations do not cover: the discrete
    model with `if_else` clamps, Delta-u bounds and a user terminal cost (Ex_NMPC_dis.py:75-77,120-125), and nx != nxp
    (Ex_LMPCxp_nlplant.py:98).  The GPU tests run the repo's own restatements of these files (examples/) against them."""
    out = {}
    for fname, tag, Ns in (("Ex_NMPC_dis.py", "nmpc_dis", 16), ("Ex_LMPCxp_nlplant.py", "lmpcxp_nlplant", 110)):
        prob = build_problem(load_example(os.path.join(REF, fname)))
        ss, ocp = make_specs(prob)
        mod = cmodel.build("ref_" + tag, prob, ocp, ss)
        rec = OracleLoop(prob, ss, ocp, mod).run(Nsim=Ns)
        print(fname, "status", rec["STATUS_DYN"], "iters", rec["ITER_DYN"])
        for key in ("U", "X_HAT", "D_HAT", "XS", "US", "Xp", "Yp", "F_DYN", "ITER_DYN", "STATUS_DYN", "STATUS_SS"):
            out["%s_%s" % (tag, key)] = rec[key]
    np.savez_compressed(os.path.join(HERE, "ref_examples_oracle.npz"), **out)


def make_problem_records(from_examples):
    """``problem_records.json``: the records of the reference files examples/ restates, or of the restatements."""
    sys.path.insert(0, os.path.dirname(HERE))
    import __graft_entry__ as entry
    from problem_record import PAIRS, RECORDS, TIMES, plain, record
    out = dict(source="examples/ restatements" if from_examples else "unmodified reference files", times=plain(TIMES),
               problems={})
    for name, fname, edits in PAIRS:
        if from_examples:
            prob, ss, ocp = entry._problem(name)
        else:
            prob = build_problem(load_example(os.path.join(REF, fname), source_edits=edits))
            ss, ocp = make_specs(prob)
        out["problems"][name] = record(prob, ss, ocp)
    with open(RECORDS, "w") as fh:
        json.dump(out, fh)


def main():
    if "--only-problem-records" in sys.argv:                      # python make_golden.py --only-problem-records
        make_problem_records("--from-examples" in sys.argv)
        return
    if not os.path.isdir(REF) and "--only-synthetic" not in " ".join(sys.argv):
        raise SystemExit("set MPC_CODE_REFERENCE to an unmodified CPCLAB-UNIPI/MPC-code checkout")
    if "--only-examples" in sys.argv:                             # python make_golden.py --only-examples
        make_reference_examples()
        return
    only = [a for a in sys.argv if a.startswith("--only-synthetic=")]
    if only:                                                      # python make_golden.py --only-synthetic=syn_12_4_20
        make_synthetic(tuple(only[0].split("=", 1)[1].split(",")))
        return
    ns = load_example(os.path.join(REF, "Ex_NMPC.py"))
    nl = load_example(os.path.join(REF, "Ex_LMPC_nlplant.py"))
    kat = dict(
        KAT1=dict(x0_m=ns["x0_m"].tolist(), u0=ns["u0"].tolist(), dhat0=ns["dhat0"].tolist(),
                  f_expected=[1.8e-7, -6.2e-4, 0.0], rk4_residual_expected=[1.5e-7, -1.1e-4, 0.0]),
        KAT2=dict(A=np.asarray(nl["A"]).tolist(), B=np.asarray(nl["B"]).tolist(), xlin=nl["xlin"].tolist(),
                  ulin=nl["ulin"].tolist(), h=nl["h"], Mx=nl["Mx"], source="Ex_LMPC_nlplant.py:85-91"),
        KAT3={"0.10": dict(xs=[0.874317, 325.000017089, 0.6528], us=[300.157302438, 0.10]),
              "0.15": dict(xs1=329.969400267, us0=296.315521811),
              "0.08": dict(xs1=322.328497426, us0=301.419219053)},
    )
    with open(os.path.join(HERE, "kat.json"), "w") as fh:
        json.dump(kat, fh, indent=1)

    prob = build_problem(ns)
    ss, ocp = make_specs(prob)
    mod = cmodel.build("ref_ex_nmpc", prob, ocp, ss)
    n, m, N = prob.nx, prob.nu, prob.N
    nxu = n + m
    rng = np.random.default_rng(12345)
    out = {}
    # ---- OCP cases: cold guess, perturbed initial state / disturbance / targets
    xs0 = np.array([0.874317, 325.000017089, 0.6528]); us0 = np.array([300.157302438, 0.1])
    cases = [(prob.x0_m, np.array([0, 0.1]), xs0, us0)]
    for i in range(7):
        xh = prob.x0_m * (1 + 0.02 * rng.uniform(-1, 1, 3))
        d = np.array([0.0, [0.1, 0.15, 0.08][i % 3]])
        xs = xs0 * (1 + 0.004 * rng.uniform(-1, 1, 3)); us = us0 * (1 + 0.004 * rng.uniform(-1, 1, 2))
        cases.append((xh, d, xs, us))
    w0 = np.zeros(ocp.nw)
    for k in range(N + 1):
        w0[nxu * k:nxu * k + n] = prob.x0_m
    for k in range(N):
        w0[nxu * k + n:nxu * (k + 1)] = prob.u0
    on = OcpNlp(ocp, mod)
    par = np.stack([np.concatenate([xh, xs, us, d, prob.u0, [0.0], np.zeros(4), np.zeros(3 * N), np.zeros(2 * N)])
                    for xh, d, xs, us in cases])
    W, F, ST, IT = [], [], [], []
    for b, (xh, d, xs, us) in enumerate(cases):
        lb, ub = ocp.w_lb.copy(), ocp.w_ub.copy()
        lb[:n] = ub[:n] = xh
        r = on.solve(w0, par[b], lb, ub, opts=IpmOptions(max_iter=100))
        W.append(r.x); F.append(r.f); ST.append(r.status); IT.append(r.iters)
        print("ocp case", b, r.return_status, r.iters, r.f)
    out.update(ocp_par=par, ocp_w0=w0, ocp_w=np.array(W), ocp_f=np.array(F), ocp_status=np.array(ST), ocp_iters=np.array(IT))
    # ---- target cases
    tn = TargetNlp(ss, mod)
    ysp, usp, xsp = [np.asarray(v, dtype=float) for v in prob.defSP(0.0)]
    dd = [np.array([0, 0.1]), np.array([0, 0.15]), np.array([0, 0.08]), np.array([0.3, 0.11]), np.array([-1.0, 0.13])]
    par_ss = np.stack([np.concatenate([usp, ysp, xsp, d, prob.u0, np.zeros(4), [0.0], np.zeros(3), np.zeros(2)]) for d in dd])
    g0 = np.stack([np.concatenate([prob.x0_m, prob.u0, mod.orc_fy(prob.x0_m, prob.u0, d, 0.0, np.zeros(2)).ravel()]) for d in dd])
    WS, FS, SS, IS = [], [], [], []
    for b in range(len(dd)):
        r = tn.solve(g0[b], par_ss[b], opts=IpmOptions(max_iter=100))
        WS.append(r.x); FS.append(r.f); SS.append(r.status); IS.append(r.iters)
        print("target case", b, r.return_status, r.iters, r.x)
    out.update(ss_par=par_ss, ss_w0=g0, ss_w=np.array(WS), ss_f=np.array(FS), ss_status=np.array(SS), ss_iters=np.array(IS))
    # ---- EKF: three consecutive updates
    P = prob.estimator["P0"].copy(); xi = np.concatenate([prob.x0_m, prob.dhat0])
    ys = np.array([[0.8745, 0.6531], [0.8751, 0.6522], [0.8739, 0.6529]])
    XI, PP = [], []
    for k in range(3):
        P, _, xi = estimators.ekf(prob, mod, ys[k], prob.u0, prob.estimator["Q"], prob.estimator["R"], P, xi, prob.h,
                                  k * prob.h, np.zeros(2), np.zeros(3))
        XI.append(xi.copy()); PP.append(P.copy())
    out.update(ekf_y=ys, ekf_xi=np.array(XI), ekf_P=np.array(PP))
    # ---- closed loop: 3 instances, 8 steps
    Bc, Ns = 3, 8
    x0 = prob.x0_p * (1 + 0.02 * np.random.default_rng(20240419).uniform(-1, 1, (Bc, 3)))
    noise = np.sqrt(1e-7) * np.random.default_rng(7).standard_normal((Ns, Bc, 2))
    loop = OracleLoop(prob, ss, ocp, mod)
    recs = [loop.run(Nsim=Ns, x0_p=x0[i], x0_m=x0[i], noise=noise[:, i, :]) for i in range(Bc)]
    out.update(cl_x0=x0, cl_noise=noise)
    for key in ("U", "X_HAT", "D_HAT", "XS", "US", "Xp", "Yp", "F_DYN", "ITER_DYN", "STATUS_DYN"):
        out["cl_" + key] = np.stack([r[key] for r in recs], axis=1)
    np.savez_compressed(os.path.join(HERE, "nmpc_oracle.npz"), **out)
    # ---- the two linear configurations: closed loop of the unmodified reference files (single instance, as shipped)
    lin = {}
    for fname, tag, Ns in (("Ex_LMPC_CSTR.py", "cstr", 24), ("Ex_LMPC_WB.py", "wb", 20), ("Ex_ENMPC.py", "enmpc", 14)):
        # Ex_ENMPC.py:109 hard-codes its estimator switch; its own EKF branch is selected (MHE is out of scope)
        edits = [("mhe_mod = 'on'", "mhe_mod = 'off'")] if tag == "enmpc" else []
        prob_l = build_problem(load_example(os.path.join(REF, fname), source_edits=edits))
        ss_l, ocp_l = make_specs(prob_l)
        mod_l = cmodel.build("ref_" + tag, prob_l, ocp_l, ss_l)
        rec = OracleLoop(prob_l, ss_l, ocp_l, mod_l).run(Nsim=Ns)
        print(fname, "status", rec["STATUS_DYN"], "iters", rec["ITER_DYN"])
        for key in ("U", "X_HAT", "D_HAT", "XS", "US", "Xp", "Yp", "F_DYN", "ITER_DYN", "STATUS_DYN", "STATUS_SS"):
            lin["%s_%s" % (tag, key)] = rec[key]
    np.savez_compressed(os.path.join(HERE, "lmpc_oracle.npz"), **lin)
    # ---- synthetic family (BASELINE configs[4]): one mid-size member whose oracle (symbolic Hessian of the unrolled
    #      RK4 graph, 8 states) takes minutes to build - hence a fixture; smaller members are checked live by the tests
    syn_args = [a for a in sys.argv if a.startswith("--synthetic")]       # --synthetic  or  --synthetic=syn_12_4_20,...
    if syn_args:
        make_synthetic(tuple(syn_args[0].split("=", 1)[1].split(",")) if "=" in syn_args[0] else ("syn_8_3_50",))
    make_reference_examples()
    make_problem_records(False)
    print("wrote fixtures")


if __name__ == "__main__":
    main()
