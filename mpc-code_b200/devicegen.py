"""Generate the per-problem device header (``mpcb_model.h``) consumed by ``csrc/mpcb_kernels.cu``.

The reference hands CasADi whole-NLP graphs and lets its VM evaluate them (``Control_Calc.py:256-258``).
Here the user's maps are emitted as small ``__device__`` functions - the continuous right-hand side
with its sensitivity / adjoint / second-order products, the output map, the stage and terminal
costs, the target problem's pieces, the plant - and the hand-written kernels orchestrate them
(RK4 sub-stepping, Riccati recursion, line search).  Matrix products that involve model Jacobians
are generated *symbolically* (e.g. ``K = f_x S + [0|f_u]``) so structural zeros cost nothing.

Layouts: matrices are column-major; symmetric matrices are packed lower-triangular row-wise
(``idx(i,j) = i(i+1)/2 + j``, ``j <= i``).
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np

from . import symbolic as S
from .codegen import CFunction, cache_expressions, emit_header, expensive_entries
from .sx import SX, Function, gradient, hessian, jacobian, mtimes, vertcat, horzcat


def tril_pack(H: SX) -> SX:
    n = H.size1()
    return SX([H[i, j]._as_scalar_expr() for i in range(n) for j in range(i + 1)]) if n else SX()


def _depends_on(expr: SX, var: SX) -> bool:
    ids = {e.uid for e in var.elements()}
    return any(s.uid in ids for s in S.symbols_of(expr.elements()))


def _cached_variants(prefix: str, base, f, vjp_in, vjp_out, sh_in, sh_out, tainted):
    """Variants of the right-hand side functions that share expensive sub-expressions between the RK4 sweeps, which
    visit the same stage points three times.  Two levels:

    * ``cache`` - transcendental values (exp, tanh, ...): computed once per stage point in sweep A (``f_c``), STORED
      in the sweeps' record, read by everything evaluated at that point later.
    * ``rc``    - reciprocals of the model's non-constant denominators (an FP64 reciprocal is ~12 instructions):
      recomputed once per stage point per sweep (``f_rc`` / ``f_rcp``) and kept in REGISTERS for the adjoint and
      second-order products at that point.  Not stored: in round 1 storing them doubled the kernel's DRAM traffic.

    Returns ``(functions, NC, NR)``; empty when the right-hand side has nothing to share."""
    consumers = [[e for _, o in vjp_out for e in SX(o).elements()], [e for _, o in sh_out for e in SX(o).elements()]]
    entries = expensive_entries(consumers, tainted, recips=True)
    if not entries:
        return [], 0, 0
    nodes = [e for e in entries if e[0] == "node"]
    recips = [e for e in entries if e[0] == "recip"]
    cache, rc = ("cache", nodes), ("rc", recips)
    fns = [CFunction(prefix + "f_c", base, [("xdot", f), ("cache", cache_expressions(nodes))]),
           CFunction(prefix + "f_rc", base, [("xdot", f), ("rc", cache_expressions(recips))], cache_in=[cache]),
           CFunction(prefix + "f_rcp", base, [("rc", cache_expressions(recips))], cache_in=[cache]),
           CFunction(prefix + "f_vjp_c", base + vjp_in, vjp_out, cache_in=[cache, rc]),
           CFunction(prefix + "f_sh_c", base + sh_in, sh_out, cache_in=[cache, rc])]
    return fns, len(nodes), len(recips)


# Above this many entries of the sensitivity block S (nx x (nx + nu)) the products of the model's derivatives with S are no
# longer generated symbolically: their size grows like nx^2 (nx + nu)^2 (26 minutes of nvcc and 266 kB of stack per thread
# for 20 states in round 1).  The generator then emits only the DENSE Jacobian and the nu-weighted Hessian of the
# right-hand side, and the device code forms K = f_x S + [0|f_u], f_x' nu and [S;E]'(nu' d2f)[S;E] with loops
# (MPCB_DENSE_SH, csrc/mpcb_device.cuh).  Override with the environment variable MPCB_DENSE_SH=0/1.
DENSE_SH_ENTRIES = 200


def _use_dense(nx: int, nu: int) -> bool:
    import os
    env = os.environ.get("MPCB_DENSE_SH")
    if env in ("0", "1"):
        return env == "1"
    return nx * (nx + nu) > DENSE_SH_ENTRIES


def _rhs_functions_dense(prefix: str, rhs: Function, nx: int, nu: int, nd: int, npx: int, nxi: int) -> List[CFunction]:
    """Right-hand side with its dense first derivatives and the adjoint-weighted Hessian (large models)."""
    x, u, d, t, px = [SX.sym(n, k) for n, k in (("x", nx), ("u", nu), ("d", nd), ("t", 1), ("px", npx))]
    f = rhs(x, u, d, t, px)
    base = [("x", x), ("u", u), ("d", d), ("t", t), ("px", px)]
    nu_adj = SX.sym("nu", nx)
    Hf, _ = hessian(mtimes(nu_adj.T, f), vertcat(x, u))
    jd = jacobian(f, d) if (nxi > nx and nd) else SX.zeros(nx, 0)
    _rhs_functions.last_cache = (0, 0)
    return [CFunction(prefix + "f", base, [("xdot", f)]),
            CFunction(prefix + "f_jac", base, [("xdot", f), ("Jx", jacobian(f, x)), ("Ju", jacobian(f, u)), ("Jd", jd)]),
            CFunction(prefix + "f_hess", base + [("nu", nu_adj)], [("M", tril_pack(Hf))])]


def _rhs_functions(prefix: str, rhs: Function, nx: int, nu: int, nd: int, npx: int, nxi: int) -> List[CFunction]:
    """Right-hand side ``f(x,u,d,t,px)`` with the products the RK4 sweeps need."""
    x, u, d, t, px = [SX.sym(n, k) for n, k in (("x", nx), ("u", nu), ("d", nd), ("t", 1), ("px", npx))]
    f = rhs(x, u, d, t, px)
    base = [("x", x), ("u", u), ("d", d), ("t", t), ("px", px)]
    fns = [CFunction(prefix + "f", base, [("xdot", f)])]
    nu_adj = SX.sym("nu", nx)
    nuf = mtimes(nu_adj.T, f)
    fns.append(CFunction(prefix + "f_vjp", base + [("nu", nu_adj)], [("fxTnu", gradient(nuf, x))]))
    fx = jacobian(f, x)
    # sensitivities with respect to (x0, u)
    nz = nx + nu
    Sxu = SX.sym("S", nx, nz)
    fu = jacobian(f, u)
    K = mtimes(fx, Sxu) + horzcat(SX.zeros(nx, nx), fu)
    fns.append(CFunction(prefix + "f_s", base + [("S", Sxu)], [("xdot", f), ("K", K)]))
    zz = vertcat(x, u)
    Hf, _ = hessian(nuf, zz)
    dZ = vertcat(Sxu, horzcat(SX.zeros(nu, nx), SX.eye(nu)))
    Hc = mtimes(dZ.T, mtimes(Hf, dZ))
    sh_out = [("xdot", f), ("K", K), ("Hc", tril_pack(Hc))]
    fns.append(CFunction(prefix + "f_sh", base + [("S", Sxu), ("nu", nu_adj)], sh_out))
    cached, nc, nr = _cached_variants(prefix, base, f, [("nu", nu_adj)], [("fxTnu", gradient(nuf, x))],
                                      [("S", Sxu), ("nu", nu_adj)], sh_out, list(nu_adj.elements()) + list(Sxu.elements()))
    fns += cached
    _rhs_functions.last_cache = (nc, nr)
    # sensitivities with respect to xi = (x0[, d]) for the estimator
    Sxi = SX.sym("S", nx, nxi)
    Kd = mtimes(fx, Sxi)
    if nxi > nx:
        Kd = Kd + horzcat(SX.zeros(nx, nx), jacobian(f, d))
    fns.append(CFunction(prefix + "f_s_xi", base + [("S", Sxi)], [("xdot", f), ("K", Kd)]))
    return fns


def _discrete_functions(prefix: str, Fx_model: Function, nx, nu, nd, npx, nxi) -> List[CFunction]:
    x, u, d, t, px = [SX.sym(n, k) for n, k in (("x", nx), ("u", nu), ("d", nd), ("t", 1), ("px", npx))]
    k = SX.sym("k", 1)
    F = Fx_model(x, u, k, d, t, px)
    if _depends_on(SX(F), k):
        raise ValueError("a discrete/linear Fx_model must not depend on the integration step k")
    base = [("x", x), ("u", u), ("d", d), ("t", t), ("px", px)]
    lam = SX.sym("lam", nx)
    zz = vertcat(x, u)
    Hf, _ = hessian(mtimes(lam.T, F), zz)
    fns = [CFunction(prefix + "F", base, [("xn", F)]),
           CFunction(prefix + "F_d", base + [("lam", lam)],
                     [("xn", F), ("A", jacobian(F, x)), ("B", jacobian(F, u)), ("Hc", tril_pack(Hf))])]
    xi = vertcat(x, d) if nxi > nx else x
    fns.append(CFunction(prefix + "F_xd", base, [("xn", F), ("Axd", jacobian(F, xi))]))
    return fns


def _sens_functions(o, D, ins_c, zz, stage_cost, rows) -> List[CFunction]:
    """Mixed second derivatives for the OCP sensitivities (csrc/mpcb_sens.cuh): derivatives of the stage gradients, the
    range rows and the terminal maps with respect to theta = [x0 | xs | us | um1] (the parameters fed in by the estimator,
    the target problem and the previous input).  ContForm: the integrated cost has no generated mixed derivatives; when
    it depends on theta the flag MPCB_SENS_CONT_DEP makes the sensitivity entry points refuse."""
    par, off, n, m = o.par, o.off, o.n, o.m
    th = vertcat(par[off["x0"]:off["us"] + m], par[off["um1"]:off["um1"] + m])
    D["MPCB_NTH"] = 2 * (n + m)
    D["MPCB_SENS_CONT_DEP"] = int(o.flags["ContForm"] is True and _depends_on(SX(o.quad_cost), th))
    gc = gradient(stage_cost, zz)
    fns = [CFunction("ocp_cost_dth", ins_c, [("Lt", jacobian(gc, th))]),
           CFunction("ocp_term_dth", [("XN", o.XN), ("par", par)], [("Tt", jacobian(gradient(o.term_cost, o.XN), th))])]
    if o.term_eq is not None:
        fns.append(CFunction("ocp_termc_dth", [("XN", o.XN), ("par", par)], [("Rt", jacobian(o.term_eq, th))]))
    if rows is not None:
        R, mult = rows
        fns.append(CFunction("ocp_out_dth", ins_c + [("mult", mult)],
                             [("Yt", jacobian(R, th)), ("HYt", jacobian(gradient(mtimes(mult.T, R), zz), th))]))
    return fns


def _sens_p_refusal(prob, o, stage_exprs) -> Optional[str]:
    """Why the sensitivities with respect to p = [d | px | py] cannot be generated for this problem, or None."""
    if o.flags["ContForm"] is True:
        return "ContForm: the integrand would need its own augmented system"
    if prob.Fx_model.meta.get("kind") == "rk4" and _use_dense(prob.nx, prob.nu):
        return "large model (dense derivative products)"
    par, off = o.par, o.off
    rest = par[off["px"]:off["end"]] if off["end"] > off["px"] else None
    if rest is not None and any(_depends_on(SX(e), rest) for e in stage_exprs):
        return "a stage or terminal map reads px / py of another stage through par"
    return None


def _sens_p_functions(prob, o, D, ins_c, zz, stage_cost, rows) -> List[CFunction]:
    """Mixed derivatives for the OCP sensitivities with respect to the parameters that enter the dynamics
    (csrc/mpcb_sens.cuh, mpcb_ocp_sens_factor_p): stage k depends on p_k = [d; px_k; py_k] only, the terminal maps on d.

    * dynamics: `_sens_model_functions`.
    * stage cost, range rows and terminal maps: as ``_sens_functions`` with respect to p_k (terminal: d).
    MPCB_SENS_P = 0 (the p entry points refuse) when `_sens_p_refusal` names a reason."""
    nd = prob.nd
    par, off = o.par, o.off
    exprs = [stage_cost, o.term_cost] + ([o.term_eq] if o.term_eq is not None else []) + ([rows[0]] if rows else [])
    why = _sens_p_refusal(prob, o, exprs)
    D["MPCB_SENS_P"] = int(why is None)
    if why is not None:
        return []
    dpar = par[off["d"]:off["d"] + nd]
    pk = vertcat(dpar, o.pxk, o.pyk)
    gc = gradient(stage_cost, zz)
    fns = [CFunction("ocp_cost_dp", ins_c, [("Lp", jacobian(gc, pk))]),
           CFunction("ocp_term_dp", [("XN", o.XN), ("par", par)], [("Tp", jacobian(gradient(o.term_cost, o.XN), dpar))])]
    if o.term_eq is not None:
        fns.append(CFunction("ocp_termc_dp", [("XN", o.XN), ("par", par)], [("Rp", jacobian(o.term_eq, dpar))]))
    if rows is not None:
        R, mult = rows
        fns.append(CFunction("ocp_out_dp", ins_c + [("mult", mult)],
                             [("Yp", jacobian(R, pk)), ("HYp", jacobian(gradient(mtimes(mult.T, R), zz), pk))]))
    model = _sens_model_functions(prob, D)
    if model is None:
        raise NotImplementedError("the map applied after the RK4 integration must be affine in (d, px)")
    return fns + model


def _sens_model_functions(prob, D) -> Optional[List[CFunction]]:
    """The model part of the sensitivities with respect to [d; px] (csrc/mpcb_sens.cuh, sens_dyn_dp), shared by the OCP
    p-blocks and the target problem's capture: dF/d[d; px] and d(grad_{x,u} lam' F)/d[d; px] of the stage map.

    * RK4: the right-hand side is integrated on the augmented state [x; q] with q' = 0, where q holds the components of
      (d, px) that the right-hand side reads (MPCB_SENS_QIDX, indices into [d; px]).  The RK4 sweeps then give dx_N/dq in
      the q columns of the sensitivity block and the mixed Hessian of lam' x_N in the packed Hessian.  The map applied
      after the integration (Bd d + px) must be affine; its Jacobian is added.  None when it is not.
    * discrete / linear: dF/d[d; px] and d(grad_{x,u} lam' F)/d[d; px] directly."""
    nx, nu, nd, npx = prob.nx, prob.nu, prob.nd, prob.npx
    fns: List[CFunction] = []
    x, u, d, t, px = [SX.sym(n, k) for n, k in (("x", nx), ("u", nu), ("d", nd), ("t", 1), ("px", npx))]
    dpx = vertcat(d, px)
    base = [("x", x), ("u", u), ("d", d), ("t", t), ("px", px)]
    if prob.Fx_model.meta.get("kind") == "rk4":
        rhs = prob.Fx_model.meta["rhs"]
        f = SX(rhs(x, u, d, t, px))
        qidx = [i for i, e in enumerate(dpx.elements()) if _depends_on(f, SX([e]))]
        D["MPCB_SENS_NQ"] = len(qidx)
        D["MPCB_SENS_QIDX"] = "{%s}" % ", ".join(str(i) for i in (qidx or [0]))
        post = SX(prob.Fx_model.meta["post"](d, px))
        Jpost = jacobian(post, dpx)
        if _depends_on(Jpost, dpx):
            return None
        fns.append(CFunction("mdl_post_dp", [("d", d), ("px", px)], [("Jp", Jpost)]))
        if qidx:
            nq = len(qidx)

            def rhs_aug(xt, u_, d_, t_, px_):
                sub = list(vertcat(d_, px_).elements())
                for j, i in enumerate(qidx):
                    sub[i] = xt[nx + j]._as_scalar_expr()
                dd, pp = SX(sub[:nd]) if nd else d_, SX(sub[nd:]) if npx else px_
                return vertcat(SX(rhs(xt[0:nx], u_, dd, t_, pp)), SX.zeros(nq, 1))

            aug = _rhs_functions("mdlp_", rhs_aug, nx + nq, nu, nd, npx, nx + nq)
            fns += [g for g in aug if g.name not in ("mdlp_f_s", "mdlp_f_s_xi")]
            D["MPCB_MDLP_NC"], D["MPCB_MDLP_NR"] = _rhs_functions.last_cache
    else:
        k = SX.sym("k", 1)
        F = SX(prob.Fx_model(x, u, k, d, t, px))
        lam = SX.sym("lam", nx)
        fns.append(CFunction("mdl_F_dp", base + [("lam", lam)],
                             [("Fp", jacobian(F, dpx)), ("Hp", jacobian(gradient(mtimes(lam.T, F), vertcat(x, u)), dpx))]))
    return fns




def _sens_tgt_functions(prob, t_, D, yres, mult, model: bool) -> List[CFunction]:
    """Mixed derivatives for the sensitivities of the target problem (csrc/mpcb_target.cuh, mpcb_target_sens_factor)
    with respect to theta_ss = [usp | ysp | xsp | d | Us_prev | px | py] (par_ss without vec(lam) and t): the cost
    gradient, and the rows after the model equalities (outputs, g_SS, h_SS) with their multiplier-weighted gradient.  The
    d / px columns of the model equalities come from `sens_dyn_dp`, whose generated functions are added here when the OCP
    p-blocks did not add them (``model``).  MPCB_SENS_TGT = 0 (the target entry points refuse) for large models on the
    dense derivative path and for a post-integration map that is not affine."""
    refused = (prob.Fx_model.meta.get("kind") == "rk4" and _use_dense(prob.nx, prob.nu)) or not D.get("MPCB_HAS_OCP")
    fns = [] if refused or not model else _sens_model_functions(prob, D)
    D["MPCB_SENS_TGT"] = int(not refused and fns is not None)
    if not D["MPCB_SENS_TGT"]:
        return []
    w, par, off = t_.wss, t_.par, t_.off
    th = par[0:off["lam"]] if off["end"] == off["px"] else vertcat(par[0:off["lam"]], par[off["px"]:off["end"]])
    D["MPCB_NTHSS"] = th.numel()
    return fns + [CFunction("tgt_cost_dth", [("w", w), ("par", par)], [("Lt", jacobian(gradient(t_.cost, w), th))]),
                  CFunction("tgt_out_dth", [("w", w), ("par", par), ("mult", mult)],
                            [("Yt", jacobian(yres, th)), ("HYt", jacobian(gradient(mtimes(mult.T, yres), w), th))])]


def generate_header(prob, ss_spec, ocp_spec, opts: Optional[Dict] = None) -> Dict[str, object]:
    """Return ``{"text": header_source, "defines": {...}, "flops": {...}}`` for one problem."""
    nx, nu, ny, nd, npx, npy, N = prob.nx, prob.nu, prob.ny, prob.nd, prob.npx, prob.npy, prob.N
    s = prob.sym
    fns: List[CFunction] = []
    D: Dict[str, object] = dict(MPCB_NX=nx, MPCB_NU=nu, MPCB_NY=ny, MPCB_ND=nd, MPCB_NPX=npx, MPCB_NPY=npy,
                                MPCB_NXP=prob.nxp, MPCB_NPXP=prob.npxp, MPCB_NPYP=prob.npyp,
                                MPCB_NH=N, MPCB_HSTEP=float(prob.h),
                                MPCB_OFFREE=0 if prob.flags["offree"] == "no" else 1,
                                MPCB_NXI=prob.nxi)
    # ---- model maps -------------------------------------------------------
    kind = prob.Fx_model.meta.get("kind")
    if kind == "rk4":
        D["MPCB_DYN_RK4"] = 1
        D["MPCB_MX"] = int(prob.Fx_model.meta["substeps"])
        dense = _use_dense(nx, nu)
        D["MPCB_DENSE_SH"] = int(dense)
        fns += (_rhs_functions_dense if dense else _rhs_functions)("mdl_", prob.Fx_model.meta["rhs"], nx, nu, nd, npx, prob.nxi)
        D["MPCB_MDL_NC"], D["MPCB_MDL_NR"] = _rhs_functions.last_cache
        d_, px_ = SX.sym("d", nd), SX.sym("px", npx)
        post = prob.Fx_model.meta["post"](d_, px_)
        fns.append(CFunction("mdl_post", [("d", d_), ("px", px_)], [("post", post), ("Jd", jacobian(post, d_))]))
    else:
        D["MPCB_DYN_RK4"] = 0
        D["MPCB_MX"] = 1
        D["MPCB_DENSE_SH"] = 0
        fns += _discrete_functions("mdl_", prob.Fx_model, nx, nu, nd, npx, prob.nxi)
    x, u, d, t, py = s["x"], s["u"], s["d"], s["t"], s["py"]
    Fy = prob.Fy_model(x, u, d, t, py)
    base_y = [("x", x), ("u", u), ("d", d), ("t", t), ("py", py)]
    xi = vertcat(x, d) if prob.flags["offree"] != "no" else x
    fns.append(CFunction("mdl_fy", base_y, [("y", Fy)]))
    fns.append(CFunction("mdl_fy_xi", base_y, [("y", Fy), ("C", jacobian(Fy, xi))]))

    # ---- plant -------------------------------------------------------------
    if prob.flags["Fp_nominal"] is True:
        D["MPCB_PLANT_NOMINAL"] = 1
        D["MPCB_PLANT_RK4"] = 0
        D["MPCB_PMX"] = 1
    else:
        D["MPCB_PLANT_NOMINAL"] = 0
        xp, pxp, pyp, pxmp, pymp, k = s["xp"], s["pxp"], s["pyp"], s["pxmp"], s["pymp"], s["k"]
        pkind = prob.Fx_p.meta.get("kind")
        if pkind == "rk4":
            D["MPCB_PLANT_RK4"] = 1
            D["MPCB_PMX"] = int(prob.Fx_p.meta["substeps"])
            rhs_p = prob.Fx_p.meta["rhs"](xp, u, pxp, t, pxmp)
            fns.append(CFunction("plt_f", [("x", xp), ("u", u), ("pxp", pxp), ("t", t), ("pxmp", pxmp)], [("xdot", rhs_p)]))
            fns.append(CFunction("plt_post", [("pxp", pxp), ("pxmp", pxmp)], [("post", prob.Fx_p.meta["post"](pxp, pxmp))]))
        else:
            D["MPCB_PLANT_RK4"] = 0
            D["MPCB_PMX"] = 1
            Fp = prob.Fx_p(xp, u, pxp, t, k, pxmp)
            if _depends_on(SX(Fp), k):
                raise ValueError("a discrete/linear plant must not depend on the integration step k")
            fns.append(CFunction("plt_F", [("x", xp), ("u", u), ("pxp", pxp), ("t", t), ("pxmp", pxmp)], [("xn", Fp)]))
        fns.append(CFunction("plt_fy", [("x", xp), ("u", u), ("pyp", pyp), ("t", t), ("pymp", pymp)],
                             [("y", prob.Fy_p(xp, u, pyp, t, pymp))]))

    # ---- OCP stage maps (Control_Calc.py:124-210) ---------------------------
    if ocp_spec is not None:
        o = ocp_spec
        if o.flags["ContForm"] is True and o.uses_uprev:
            raise NotImplementedError("ContForm together with Delta-u terms is not on the device path")
        if o.flags["ContForm"] is True and D.get("MPCB_DENSE_SH"):
            raise NotImplementedError("ContForm is not available for large models (dense derivative products)")
        if o.term_eq is not None:                       # TermCons: X_N - x_s = 0 (X_N = 0 without QForm), Control_Calc.py:194-198
            Jt = jacobian(o.term_eq, o.XN)
            ident = all((e.op == "const" and float(e.val) == (1.0 if i % (o.n + 1) == 0 else 0.0)) for i, e in enumerate(Jt.elements()))
            if not ident:
                raise NotImplementedError("terminal equality must have the form X_N - const")
        # Delta-u costs / bounds couple u_k with u_{k-1} (Control_Calc.py:163-169,180-183): the device carries
        # u_{k-1} as extra state components v_k (z_k = [x_k; v_k], v_{k+1} = u_k), so every stage map stays local.
        naug = m_ = o.m if o.uses_uprev else 0
        n_rows = (0 if o.yFree else o.p) + (0 if o.DuFree else o.m) + o.n_gin
        D.update(MPCB_HAS_OCP=1, MPCB_NW=o.nw, MPCB_NPAR=o.npar, MPCB_NG=n_rows, MPCB_NAUG=naug,
                 MPCB_NGY=(0 if o.yFree else o.p), MPCB_NGDU=(0 if o.DuFree else o.m), MPCB_NGIN=o.n_gin)
        for k_, v_ in o.off.items():
            D["MPCB_OFF_%s" % k_.upper()] = v_
        X, U, Up, par, pxk, pyk = o.X, o.U, o.Uprev, o.par, o.pxk, o.pyk
        Z = vertcat(X, Up) if naug else X               # stage state seen by the kernels
        zz = vertcat(Z, U)
        ins_c = [("Z", Z), ("U", U), ("par", par), ("pxk", pxk), ("pyk", pyk)]
        if o.flags["ContForm"] is True:
            # stage cost = quadrature state of the integrator (Control_Calc.py:102-111,153-158): the right-hand side
            # [fx + px; F_obj] on the state [x; q] with the products the RK4 sweeps need; ocp_cost* are then zero.
            D.update(MPCB_CONTFORM=1, MPCB_CMX=int(o.cont_substeps))
            q = SX.sym("q", 1)
            xt = vertcat(X, q)
            rhs_t = vertcat(SX(o.cont_rhs), SX(o.quad_cost))
            ns = o.n + 1
            base_q = [("xt", xt), ("U", U), ("par", par), ("pxk", pxk), ("pyk", pyk)]
            nu_adj = SX.sym("nu", ns)
            nuf = mtimes(nu_adj.T, rhs_t)
            St = SX.sym("S", ns, ns + o.m)
            Kt = mtimes(jacobian(rhs_t, xt), St) + horzcat(SX.zeros(ns, ns), jacobian(rhs_t, U))
            Hft, _ = hessian(nuf, vertcat(xt, U))
            dZt = vertcat(St, horzcat(SX.zeros(o.m, ns), SX.eye(o.m)))
            sh_out = [("xdot", rhs_t), ("K", Kt), ("Hc", tril_pack(mtimes(dZt.T, mtimes(Hft, dZt))))]
            fns.append(CFunction("ocq_f", base_q, [("xdot", rhs_t)]))
            fns.append(CFunction("ocq_f_vjp", base_q + [("nu", nu_adj)], [("fxTnu", gradient(nuf, xt))]))
            fns.append(CFunction("ocq_f_sh", base_q + [("S", St), ("nu", nu_adj)], sh_out))
            cached, nc, nr = _cached_variants("ocq_", base_q, rhs_t, [("nu", nu_adj)], [("fxTnu", gradient(nuf, xt))],
                                              [("S", St), ("nu", nu_adj)], sh_out, list(nu_adj.elements()) + list(St.elements()))
            fns += cached
            D["MPCB_OCQ_NC"], D["MPCB_OCQ_NR"] = nc, nr
            stage_cost = SX(0.0)
        else:
            D.update(MPCB_CONTFORM=0, MPCB_CMX=1)
            stage_cost = o.stage_cost
        Hc, gc = hessian(stage_cost, zz)
        fns.append(CFunction("ocp_cost", ins_c, [("l", stage_cost)]))
        fns.append(CFunction("ocp_cost_d", ins_c, [("l", stage_cost), ("g", gc), ("H", tril_pack(Hc))]))
        D["MPCB_TERMCONS"] = int(o.term_eq is not None)
        if o.term_eq is not None:
            fns.append(CFunction("ocp_termc", [("XN", o.XN), ("par", par)], [("r", o.term_eq)]))
        Ht, gt = hessian(o.term_cost, o.XN)
        fns.append(CFunction("ocp_term", [("XN", o.XN), ("par", par)], [("V", o.term_cost)]))
        fns.append(CFunction("ocp_term_d", [("XN", o.XN), ("par", par)],
                             [("V", o.term_cost), ("g", gt), ("H", tril_pack(Ht))]))
        if n_rows:
            rows = []
            if not o.yFree:
                rows.append(o.Y)
            if not o.DuFree:
                rows.append(o.DU)
            if o.G is not None:                         # user stage inequalities, after the Y and DU rows
                rows.append(o.G)
            R = vertcat(*rows)
            mult = SX.sym("mult", n_rows)
            Hy, _ = hessian(mtimes(mult.T, R), zz)
            ins_y = [("Z", Z), ("U", U), ("par", par), ("pxk", pxk), ("pyk", pyk)]
            fns.append(CFunction("ocp_out", ins_y, [("Y", R)]))
            fns.append(CFunction("ocp_out_d", ins_y + [("mult", mult)],
                                 [("Y", R), ("JY", jacobian(R, zz)), ("HY", tril_pack(Hy))]))
            D["MPCB_OUT_LINEAR"] = int(all(e is S.ZERO for e in Hy.elements()))
        fns += _sens_functions(o, D, ins_c, zz, stage_cost, rows=(R, mult) if n_rows else None)
        fns += _sens_p_functions(prob, o, D, ins_c, zz, stage_cost, rows=(R, mult) if n_rows else None)
    else:
        D["MPCB_HAS_OCP"] = 0

    # ---- target problem (Target_Calc.py:75-124) ------------------------------
    if ss_spec is not None:
        t_ = ss_spec
        D.update(MPCB_HAS_TARGET=1, MPCB_NWSS=t_.nw, MPCB_NPARSS=t_.npar, MPCB_NGSS=t_.ng_ss, MPCB_NHSS=t_.nh_ss)
        for k_, v_ in t_.off.items():
            D["MPCB_OFFSS_%s" % k_.upper()] = v_
        w, par = t_.wss, t_.par
        Hf, gf = hessian(t_.cost, w)
        fns.append(CFunction("tgt_cost", [("w", w), ("par", par)], [("f", t_.cost)]))
        fns.append(CFunction("tgt_cost_d", [("w", w), ("par", par)], [("f", t_.cost), ("g", gf), ("H", tril_pack(Hf))]))
        # rows after the model equalities: output map, then the user rows g_SS <= 0 and h_SS = 0 (Target_Calc.py:80-109)
        yres = t_.Ynext - t_.Ys
        if t_.Gss is not None:
            yres = vertcat(yres, t_.Gss)
        if t_.Hss is not None:
            yres = vertcat(yres, t_.Hss)
        yres = SX(yres)
        mult = SX.sym("mult", yres.numel())
        Hy, _ = hessian(mtimes(mult.T, yres), w)
        fns.append(CFunction("tgt_out", [("w", w), ("par", par)], [("r", yres)]))
        fns.append(CFunction("tgt_out_d", [("w", w), ("par", par), ("mult", mult)],
                             [("r", yres), ("J", jacobian(yres, w)), ("H", tril_pack(Hy))]))
        fns += _sens_tgt_functions(prob, t_, D, yres, mult, model=not D.get("MPCB_SENS_P"))
    else:
        D["MPCB_HAS_TARGET"] = 0

    for f in fns:
        f.shared_reciprocals = True          # device code only; the oracle's generated C keeps true divisions
    flops = {f.name: f.flops for f in fns}
    table = " ".join('{"%s", %dL},' % (n, v) for n, v in flops.items())
    text = emit_header("MPCB_MODEL_H", D, fns, preamble="#define MPCB_FLOPS_TABLE " + table)
    return dict(text=text, defines=D, flops=flops, functions=fns)
