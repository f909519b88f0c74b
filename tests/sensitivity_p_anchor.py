"""Active-set anchor for the OCP sensitivities with respect to p = [d | px_0..px_{N-1} | py_0..py_{N-1}], the parameters
that enter the dynamics (TEST INFRASTRUCTURE, tests/test_ocp_sensitivity_params.py).

The p counterpart of ``oracle/sensitivity.py``: at an oracle solution the bounds and range rows are classified by their
distance to the bound, the active ones are fixed, and the dense equality-constrained KKT system of the NLP of
`oracle.nlp.OcpNlp` is solved with NumPy,

    [H   J_A'] [dw ]     [d(grad_w L)/dp]
    [J_A  0  ] [dlam] = -[d(g_A)/dp     ]      (dw_i = 0 on active bounds),   L = f + lam' g.

p enters the dynamics, so the rows F_k - X_{k+1} of the dynamics have the non-zero right-hand sides dF_k/dp: ordinary rows
of d(g_A)/dp.  The mixed derivatives are symbolic (the unrolled stage expressions of the OCP spec, differentiated with the
tracer and compiled to C like `oracle.cmodel` does).
"""
from __future__ import annotations

import numpy as np

from mpc_code_b200.codegen import CFunction, CModule
from mpc_code_b200.sx import SX, gradient, jacobian, mtimes, vertcat
from oracle.cmodel import BUILD_DIR


def _active_set(nlp, w, lam, par, w_lb, w_ub, g_lb, g_ub, gap, act):
    """Hessian, constraint Jacobian, fixed bounds and active rows at (w, lam), and whether the active set is clear."""
    s = nlp.s
    n = s.n
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
    return H, J, fixed, rows, clear


def _active_set_solve(H, J, fixed, rows, Lt, Gt):
    """dw [nw, ncols] of the equality-constrained KKT system with the fixed bounds eliminated and the rows `rows` active,
    and whether that system is regular (else its least-squares solution is returned)."""
    free = np.where(~fixed)[0]
    JA = J[np.ix_(rows, free)]
    nf, na = free.size, len(rows)
    K = np.zeros((nf + na, nf + na))
    K[:nf, :nf] = H[np.ix_(free, free)]; K[:nf, nf:] = JA.T; K[nf:, :nf] = JA
    rhs = -np.vstack([Lt[free], Gt[rows]])
    regular = np.linalg.matrix_rank(K) == K.shape[0]
    sol = np.linalg.solve(K, rhs) if regular else np.linalg.lstsq(K, rhs, rcond=None)[0]
    dW = np.zeros((H.shape[0], Lt.shape[1]))
    dW[free] = sol[:nf]
    return dW, regular


def param_count(spec):
    return spec.nd + (spec.npx + spec.npy) * spec.N


def param_index(spec, k, c):
    """Index into p of column c of p_k = [d; px_k; py_k]."""
    nd, npx, npy, N = spec.nd, spec.npx, spec.npy, spec.N
    if c < nd:
        return c
    if c < nd + npx:
        return nd + k * npx + (c - nd)
    return nd + npx * N + k * npy + (c - nd - npx)


def build_p(name, spec) -> CModule:
    """Mixed derivatives of one stage of the OCP Lagrangian, of its rows and of the terminal maps with respect to
    p_k = [d; px_k; py_k] (terminal: d)."""
    X, U, Up, par, pxk, pyk = spec.X, spec.U, spec.Uprev, spec.par, spec.pxk, spec.pyk
    n, p, off = spec.n, spec.p, spec.off
    dpar = par[off["d"]:off["d"] + spec.nd]
    pk = vertcat(dpar, pxk, pyk)
    lam, mult = SX.sym("lam", n), SX.sym("mult", max(p, 1))
    L = spec.stage_cost + mtimes(lam.T, spec.Xnext)
    outs_g = [("Fp", jacobian(spec.Xnext, pk)), ("Yp", jacobian(spec.Y, pk) if p else SX.zeros(1, pk.numel()))]
    if p:
        L = L + mtimes(mult[0:p].T, spec.Y)
    ins = [("X", X), ("U", U), ("Up", Up), ("par", par), ("pxk", pxk), ("pyk", pyk), ("lam", lam), ("mult", mult)]
    if getattr(spec, "G", None) is not None:
        multg = SX.sym("multg", spec.G.numel())
        L = L + mtimes(multg.T, spec.G)
        ins.append(("multg", multg))
        outs_g.append(("Gp", jacobian(spec.G, pk)))
    gz = gradient(L, vertcat(X, U, Up))
    term = [("Tp", jacobian(gradient(spec.term_cost, spec.XN), dpar))]
    if spec.term_eq is not None:
        term.append(("Rp", jacobian(spec.term_eq, dpar)))
    fns = [CFunction("sens_stage_p", ins, [("Lp", jacobian(gz, pk))] + outs_g),
           CFunction("sens_term_p", [("XN", spec.XN), ("par", par)], term)]
    return CModule("orc_sensp_" + name, fns, BUILD_DIR)


def mixed_blocks_p(nlp, smod, w, lam, par):
    """d(grad_w L)/dp [nw, n_p] and dg/dp [m, n_p] of `nlp` (an OcpNlp) at (w, lam); smod from `build_p`."""
    s = nlp.s
    n, p, N, nxu = s.n, s.p, s.N, nlp.nxu
    par = np.asarray(par, dtype=float).reshape(-1)
    npk = s.nd + s.npx + s.npy
    Lt = np.zeros((s.nw, param_count(s))); Gt = np.zeros((nlp.m_total, param_count(s)))
    um1 = par[s.off["um1"]:s.off["um1"] + s.m]
    oy, ogi, ngi = nlp.n_dyn, nlp.n_dyn + nlp.n_y + nlp.n_du, nlp.n_gin
    for k in range(N):
        cols = [param_index(s, k, c) for c in range(npk)]
        X = w[nxu * k:nxu * k + n]; U = w[nxu * k + n:nxu * (k + 1)]
        Up = um1 if k == 0 else w[nxu * (k - 1) + n:nxu * k]
        pxk, pyk = nlp._slices(par, k)
        rows = slice(n * (k + 1), n * (k + 2))
        mult = lam[oy + p * k:oy + p * (k + 1)] if nlp.n_y else np.zeros(max(p, 1))
        args = [X, U, Up, par, pxk, pyk, lam[rows], mult]
        if ngi:
            args.append(lam[ogi + ngi * k:ogi + ngi * (k + 1)])
        out = smod.sens_stage_p(*args)
        Lp, Fp, Yp = out[:3]
        Lt[nxu * k:nxu * (k + 1), cols] += Lp[:nxu]
        if k > 0:                                                          # U_{-1} = um1 is not a function of p
            Lt[nxu * (k - 1) + n:nxu * k, cols] += Lp[nxu:]
        Gt[rows, cols] += Fp
        if nlp.n_y:
            Gt[oy + p * k:oy + p * (k + 1), cols] += Yp
        if ngi:
            Gt[ogi + ngi * k:ogi + ngi * (k + 1), cols] += out[3]
    out = smod.sens_term_p(w[nxu * N:nxu * N + n], par)
    nd = s.nd
    Lt[nxu * N:nxu * N + n, :nd] += out[0]
    if s.term_eq is not None:
        Gt[n * (N + 1):n * (N + 2), :nd] += out[1]
    return Lt, Gt


def active_set_jacobian_p(nlp, smod, res, par, w_lb, w_ub, g_lb, g_ub, gap=1e-4, act=1e-6):
    """dw*/dp [nw, n_p] of the oracle solution ``res`` and whether its active set is clear (as `active_set_jacobian`)
    with linearly independent active constraints: an active output row that restates an active bound leaves the
    derivative along its offset py undetermined."""
    w, lam = np.asarray(res.x, dtype=float), np.asarray(res.lam_g, dtype=float)
    H, J, fixed, rows, clear = _active_set(nlp, w, lam, par, w_lb, w_ub, g_lb, g_ub, gap, act)
    Lt, Gt = mixed_blocks_p(nlp, smod, w, lam, par)
    dW, regular = _active_set_solve(H, J, fixed, rows, Lt, Gt)
    return dW, bool(clear and regular)
