"""Active-set anchor for the sensitivities of the steady-state target problem (TEST INFRASTRUCTURE,
tests/test_target_sensitivity.py).

theta_ss = [usp | ysp | xsp | d | Us_prev | px | py] is par_ss without vec(lam) and t.  At an oracle solution of
`oracle.nlp.TargetNlp` the bounds and the inequality rows are classified by their distance to the bound, the active ones
are fixed, and the dense equality-constrained KKT system is solved with NumPy,

    [H   J_A'] [dw ]     [d(grad_w L)/dtheta_ss]
    [J_A  0  ] [dlam] = -[d(g_A)/dtheta_ss     ]      (dw_i = 0 on active bounds),   L = f + lam' g.

The mixed derivatives are symbolic: the target spec's expressions, differentiated with the tracer and compiled to C like
`oracle.cmodel` does.
"""
from __future__ import annotations

import numpy as np

from mpc_code_b200.codegen import CFunction, CModule
from mpc_code_b200.sx import SX, gradient, jacobian, mtimes, vertcat
from oracle.cmodel import BUILD_DIR
from sensitivity_p_anchor import _active_set_solve


def theta_ss_index(ss):
    """Indices into par_ss of the components of theta_ss."""
    off = ss.off
    return list(range(0, off["lam"])) + list(range(off["px"], off["end"]))


def _constraints(ss):
    con = vertcat(ss.Xnext - ss.Xs, ss.Ynext - ss.Ys)
    for extra in (ss.Gss, ss.Hss):
        if extra is not None:
            con = vertcat(con, extra)
    return SX(con)


def build(name, ss) -> CModule:
    """d(grad_w L)/dtheta_ss and dg/dtheta_ss of the target NLP, with its constraint vector in the oracle's order."""
    par = ss.par
    th = SX([par[i]._as_scalar_expr() for i in theta_ss_index(ss)])
    con = _constraints(ss)
    mult = SX.sym("mult", con.numel())
    L = ss.cost + mtimes(mult.T, con)
    fns = [CFunction("tgt_sens", [("w", ss.wss), ("par", par), ("mult", mult)],
                     [("Lt", jacobian(gradient(L, ss.wss), th)), ("Gt", jacobian(con, th))])]
    return CModule("orc_senstgt_" + name, fns, BUILD_DIR)


def active_set_jacobian(nlp, smod, res, par, gap=1e-4, act=1e-6):
    """dwss*/dtheta_ss [nw, ntheta_ss] of the oracle solution ``res`` and whether its active set is clear: every bound and
    inequality row either inactive with a distance > ``gap`` or at distance < ``act`` with a multiplier of magnitude
    > ``act``, and the active constraints linearly independent."""
    s = nlp.s
    w, lam = np.asarray(res.x, dtype=float), np.asarray(res.lam_g, dtype=float)
    ev = nlp.make_fun(par)(w, lam, 2)
    H, J, g = ev["H"], ev["J"], ev["g"]
    rgrad = ev["grad"] + J.T @ lam                                         # reduced gradient = bound multipliers zU - zL
    clear = True
    fixed = np.zeros(s.nw, dtype=bool)
    for i in range(s.nw):
        dist = min(abs(w[i] - s.w_lb[i]), abs(s.w_ub[i] - w[i]))
        if dist < act:
            fixed[i] = True
            clear &= abs(rgrad[i]) > act
        else:
            clear &= dist > gap
    rows = []
    for r in range(g.size):
        if s.g_lb[r] == s.g_ub[r]:
            rows.append(r)
            continue
        dist = min(abs(g[r] - s.g_lb[r]), abs(s.g_ub[r] - g[r]))
        if dist < act:
            rows.append(r)
            clear &= abs(lam[r]) > act
        else:
            clear &= dist > gap
    Lt, Gt = smod.tgt_sens(w, np.asarray(par, dtype=float), lam)
    dW, regular = _active_set_solve(H, J, fixed, rows, Lt, Gt)
    return dW, bool(clear and regular)
