"""Active-set anchor for the OCP sensitivities (TEST INFRASTRUCTURE - see ``oracle/__init__.py``).

At an oracle solution the bounds and range rows are classified by their distance to the bound; the active ones are
fixed and the dense equality-constrained KKT system of the NLP of `oracle.nlp.OcpNlp` is solved with NumPy:

    [H   J_A'] [dw ]     [d(grad_w L)/dtheta]
    [J_A  0  ] [dlam] = -[d(g_A)/dtheta     ]      (dw_i = 0 on active bounds),   L = f + lam' g.

The mixed derivatives d(grad_w L)/dtheta and dg/dtheta are SYMBOLIC: the unrolled stage expressions of the OCP spec
are differentiated with the tracer and compiled to C like `oracle.cmodel` does (no finite differences, no complex step).
theta = [x0 | xs | us | um1] as in ``include/mpcb.h``.
"""
from __future__ import annotations

import numpy as np

from mpc_code_b200.codegen import CFunction, CModule
from mpc_code_b200.sx import SX, gradient, jacobian, mtimes, vertcat

from .cmodel import BUILD_DIR


def theta_symbols(spec):
    par, off, m = spec.par, spec.off, spec.m
    return vertcat(par[off["x0"]:off["us"] + m], par[off["um1"]:off["um1"] + m])


def build(name, spec) -> CModule:
    """Mixed derivatives of one stage of the OCP Lagrangian and of the terminal cost with respect to theta."""
    X, U, Up, par, pxk, pyk = spec.X, spec.U, spec.Uprev, spec.par, spec.pxk, spec.pyk
    n, p = spec.n, spec.p
    th = theta_symbols(spec)
    lam, mult = SX.sym("lam", n), SX.sym("mult", max(p, 1))
    L = spec.stage_cost + mtimes(lam.T, spec.Xnext)
    outs_g = [("Fp", jacobian(spec.Xnext, th)), ("Yp", jacobian(spec.Y, th) if p else SX.zeros(1, th.numel()))]
    if p:
        L = L + mtimes(mult[0:p].T, spec.Y)
    ins = [("X", X), ("U", U), ("Up", Up), ("par", par), ("pxk", pxk), ("pyk", pyk), ("lam", lam), ("mult", mult)]
    if getattr(spec, "G", None) is not None:
        multg = SX.sym("multg", spec.G.numel())
        L = L + mtimes(multg.T, spec.G)
        ins.append(("multg", multg))
        outs_g.append(("Gp", jacobian(spec.G, th)))
    gz = gradient(L, vertcat(X, U, Up))
    fns = [CFunction("sens_stage", ins, [("Lp", jacobian(gz, th)), ("Lup", jacobian(gz, Up))] + outs_g),
           CFunction("sens_term", [("XN", spec.XN), ("par", par)],
                     [("Tp", jacobian(gradient(spec.term_cost, spec.XN), th))])]
    return CModule("orc_sens_" + name, fns, BUILD_DIR)


def mixed_blocks(nlp, smod, w, lam, par):
    """d(grad_w L)/dtheta [nw, ntheta] and dg/dtheta [m, ntheta] of `nlp` (an OcpNlp) at (w, lam)."""
    s = nlp.s
    n, m, p, N, nxu = s.n, s.m, s.p, s.N, nlp.nxu
    par = np.asarray(par, dtype=float).reshape(-1)
    nth = 2 * (n + m)
    ix0, ixs, ium1 = slice(0, n), slice(n, 2 * n), slice(2 * n + m, nth)
    Lt = np.zeros((s.nw, nth)); Gt = np.zeros((nlp.m_total, nth))
    Gt[0:n, ix0] = np.eye(n)                                              # x0 - X_0
    um1 = par[s.off["um1"]:s.off["um1"] + m]
    oy, odu, ogi, ngi = nlp.n_dyn, nlp.n_dyn + nlp.n_y, nlp.n_dyn + nlp.n_y + nlp.n_du, nlp.n_gin
    for k in range(N):
        X = w[nxu * k:nxu * k + n]; U = w[nxu * k + n:nxu * (k + 1)]
        Up = um1 if k == 0 else w[nxu * (k - 1) + n:nxu * k]
        pxk, pyk = nlp._slices(par, k)
        rows = slice(n * (k + 1), n * (k + 2))
        mult = lam[oy + p * k:oy + p * (k + 1)] if nlp.n_y else np.zeros(max(p, 1))
        args = [X, U, Up, par, pxk, pyk, lam[rows], mult]
        if ngi:
            args.append(lam[ogi + ngi * k:ogi + ngi * (k + 1)])
        out = smod.sens_stage(*args)
        Lp, Lup, Fp, Yp = out[:4]
        iz = slice(nxu * k, nxu * (k + 1))
        Lt[iz] += Lp[:nxu]
        if k > 0:
            Lt[nxu * (k - 1) + n:nxu * k] += Lp[nxu:]
        else:                                                              # U_{-1} = um1 is a parameter
            Lt[iz, ium1] += Lup[:nxu]
        Gt[rows] = Fp
        if nlp.n_y:
            Gt[oy + p * k:oy + p * (k + 1)] = Yp
        if nlp.n_du and k == 0:
            Gt[odu:odu + m, ium1] = -np.eye(m)                             # U_0 - um1
        if ngi:
            Gt[ogi + ngi * k:ogi + ngi * (k + 1)] = out[4]
    Lt[nxu * N:nxu * N + n] += smod.sens_term(w[nxu * N:nxu * N + n], par)
    if s.term_eq is not None and s.flags["QForm"]:
        Gt[n * (N + 1):n * (N + 2), ixs] = -np.eye(n)                     # X_N - xs
    return Lt, Gt


def active_set_jacobian(nlp, smod, res, par, w_lb, w_ub, g_lb, g_ub, gap=1e-4, act=1e-6):
    """dw*/dtheta [nw, ntheta] of the oracle solution ``res`` by the active-set KKT system, and whether the active set is
    clear: every bound / range row either inactive with a distance > ``gap`` or at distance < ``act`` with a multiplier
    of magnitude > ``act`` (strongly active)."""
    s = nlp.s
    n = s.n
    w, lam = np.asarray(res.x, dtype=float), np.asarray(res.lam_g, dtype=float)
    fun = nlp.make_fun(par)
    ev = fun(w, lam, 2)
    H, J, g = ev["H"], ev["J"], ev["g"]
    rgrad = ev["grad"] + J.T @ lam                                         # reduced gradient = bound multipliers zU - zL
    clear = True
    fixed = np.zeros(s.nw, dtype=bool)
    for i in range(n, s.nw):
        dist = min(abs(w[i] - w_lb[i]), abs(w_ub[i] - w[i]))
        if dist < act:
            fixed[i] = True
            clear &= abs(rgrad[i]) > act
        else:
            clear &= dist > gap
    rows = []
    for r in range(g.size):
        if g_lb[r] == g_ub[r]:
            rows.append(r)
            continue
        dist = min(abs(g[r] - g_lb[r]), abs(g_ub[r] - g[r]))
        if dist < act:
            rows.append(r)
            clear &= abs(lam[r]) > act
        else:
            clear &= dist > gap
    Lt, Gt = mixed_blocks(nlp, smod, w, lam, par)
    free = np.where(~fixed)[0]
    JA = J[np.ix_(rows, free)]
    nf, na = free.size, len(rows)
    K = np.zeros((nf + na, nf + na))
    K[:nf, :nf] = H[np.ix_(free, free)]; K[:nf, nf:] = JA.T; K[nf:, :nf] = JA
    rhs = -np.vstack([Lt[free], Gt[rows]])
    sol = np.linalg.lstsq(K, rhs, rcond=None)[0] if np.linalg.matrix_rank(K) < K.shape[0] else np.linalg.solve(K, rhs)
    dW = np.zeros((s.nw, Lt.shape[1]))
    dW[free] = sol[:nf]
    return dW, bool(clear)
