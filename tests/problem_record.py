"""TEST INFRASTRUCTURE: everything that defines one MPC problem, as plain JSON data - dimensions, flags, model / plant /
output maps and costs evaluated at seeded random points, set-points, parameters, bounds, parameter offsets, estimator
data and initial state.  ``tests/golden/problem_records.json`` holds the records of the reference's ``Ex_*.py`` files
(``tests/golden/make_golden.py --only-problem-records``); the tests compare the records of the restatements under
``examples/`` with them, so that those tests need no reference checkout."""
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
RECORDS = os.path.join(HERE, "golden", "problem_records.json")

# example under examples/ -> reference file it restates, and the source edits applied to that file when it is loaded
# (Ex_ENMPC.py:109 hard-codes its estimator switch; its own EKF branch is selected, MHE is out of scope)
PAIRS = [("nmpc_cstr", "Ex_NMPC.py", ()), ("lmpc_cstr", "Ex_LMPC_CSTR.py", ()), ("lmpc_wb", "Ex_LMPC_WB.py", ()),
         ("lmpc_nlplant", "Ex_LMPC_nlplant.py", ()), ("nmpc_dis", "Ex_NMPC_dis.py", ()),
         ("lmpcxp_nlplant", "Ex_LMPCxp_nlplant.py", ()),
         ("enmpc_reactor", "Ex_ENMPC.py", (("mhe_mod = 'on'", "mhe_mod = 'off'"),))]
DIMS = ("nx", "nxp", "nu", "ny", "nd", "N", "Nsim", "h", "npx", "npy", "npxp", "npyp", "nxi")
TIMES = (0.0, 4.9, 19.9, 20.0, 25.0, 50.0, 55.0, 1500.0, 2250.0, 2251.0, 4500.0, 6000.0)
PARAM_FNS = ("def_px", "def_py", "def_pxp", "def_pyp", "def_pxmp", "def_pymp")


def plain(v):
    """JSON-ready copy of ``v`` (numpy arrays and scalars become lists and Python numbers)."""
    if isinstance(v, dict):
        return {str(k): plain(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [plain(x) for x in v]
    if v is None or isinstance(v, (bool, str)):
        return v
    if isinstance(v, (np.bool_,)):
        return bool(v)
    if isinstance(v, (int, np.integer)):
        return int(v)
    if isinstance(v, (float, np.floating)):
        return float(v)
    return np.asarray(v, dtype=float).tolist()


def points(prob):
    """Four seeded evaluation points around the problem's initial state (inputs of every map in the record)."""
    rng = np.random.default_rng(0)
    nx, nxp, nu, ny, nd = prob.nx, prob.nxp, prob.nu, prob.ny, prob.nd
    out = []
    for _ in range(4):
        x = prob.x0_m * (1 + 0.02 * rng.standard_normal(nx)) + 1e-3 * rng.standard_normal(nx)
        xp = prob.x0_p * (1 + 0.02 * rng.standard_normal(nxp)) + 1e-3 * rng.standard_normal(nxp)
        u = prob.u0 * (1 + 0.01 * rng.standard_normal(nu)) + 1e-3 * rng.standard_normal(nu)
        d = 0.1 * rng.standard_normal(nd); t = float(rng.uniform(0, 30))
        px, py = 1e-3 * rng.standard_normal(prob.npx), 1e-3 * rng.standard_normal(prob.npy)
        pxp, pyp = 1e-3 * rng.standard_normal(prob.npxp), 1e-3 * rng.standard_normal(prob.npyp)
        if prob.flags["offree"] == "nl":
            d = np.abs(d) + 0.05                      # a physical feed rate for the CSTR models
        y = rng.standard_normal(ny); xs = rng.standard_normal(nx); us = rng.standard_normal(nu); ys = rng.standard_normal(ny)
        out.append(dict(x=x, xp=xp, u=u, d=d, t=t, px=px, py=py, pxp=pxp, pyp=pyp, y=y, xs=xs, us=us, ys=ys))
    return out


def evaluate(prob, pt):
    """The problem's maps and costs at one point (``pt`` as made by ``points``, or as read back from a record)."""
    a = {k: (v if k == "t" else np.asarray(v, dtype=float)) for k, v in pt.items()}
    x, xp, u, d, t, h = a["x"], a["xp"], a["u"], a["d"], a["t"], prob.h
    ev = lambda v: np.asarray(v, dtype=float).tolist()  # noqa: E731
    return dict(Fx_model=ev(prob.Fx_model(x, u, h, d, t, a["px"])), Fy_model=ev(prob.Fy_model(x, u, d, t, a["py"])),
                Fx_p=ev(prob.Fx_p(xp, u, a["pxp"], t, h, a["pxp"])), Fy_p=ev(prob.Fy_p(xp, u, a["pyp"], t, a["pyp"])),
                F_obj=ev(prob.F_obj(x, u, a["y"], a["xs"], a["us"], a["ys"])),
                Fss_obj=ev(prob.Fss_obj(x, u, a["y"], a["xs"], a["us"], a["ys"])), Vfin=ev(prob.Vfin(x, a["xs"])))


def record(prob, ss, ocp):
    """The JSON-ready record of one problem and its target / OCP specs (``make_specs``)."""
    rec = {attr: plain(getattr(prob, attr)) for attr in DIMS}
    rec.update(flags=plain(prob.flags), sol_optss=plain(prob.sol_optss), sol_optdyn=plain(prob.sol_optdyn),
               R_wn=plain(prob.R_wn))
    for attr in ("x0_p", "x0_m", "u0", "dhat0"):
        rec[attr] = plain(getattr(prob, attr))
    pts = points(prob)
    rec["points"] = [plain(pt) for pt in pts]
    rec["evals"] = [evaluate(prob, pt) for pt in pts]
    rec["defSP"] = None if prob.defSP is None else [plain(list(prob.defSP(t))) for t in TIMES]
    rec["params"] = {fn: [plain(prob.ns[fn](t)[0]) for t in TIMES] for fn in PARAM_FNS if fn in prob.ns}
    for tag, spec in (("ocp", ocp), ("ss", ss)):
        rec[tag] = {k: plain(getattr(spec, k)) for k in ("w_lb", "w_ub", "g_lb", "g_ub", "off")}
    rec["ocp"].update(flags=plain(ocp.flags), yFree=plain(ocp.yFree), DuFree=plain(ocp.DuFree), uses_uprev=plain(ocp.uses_uprev))
    est = prob.estimator
    rec["estimator"] = dict(type=est["type"], **{k: plain(est.get(k)) for k in ("Q", "R", "K", "P0", "dmin", "dmax")})
    return rec


def load_records():
    with open(RECORDS) as fh:
        return json.load(fh)
