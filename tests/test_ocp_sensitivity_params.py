"""Sensitivities of the batched OCP solution with respect to p = [d | px_0..px_{N-1} | py_0..py_{N-1}], the parameters
that enter the dynamics (csrc/mpcb_sens.cuh, mpcb_ocp_sens_factor_p / mpcb_ocp_jvp_p / mpcb_ocp_vjp_p).

Without a GPU the device arithmetic runs on the CPU through tests/cpu_harness_sens_p.cpp and is checked against the
active-set anchor of tests/sensitivity_p_anchor.py (itself checked against finite differences of the oracle solve),
against the condensed least-squares solution of an unconstrained linear MPC in NumPy, and for adjoint consistency.  The `-m gpu`
tests repeat the comparisons through the C ABI and the Python layer on the device.
"""
import ctypes

import numpy as np
import pytest

from conftest import _bundle
from test_ocp_sensitivity import G, TIGHT, _col_close, _device_solver, _nmpc_batch, oracle_solve, sample_pars, \
    sens_harness

VP = ctypes.c_void_p
_SENS_P_HARNESS = {}


def sens_p_harness(b):
    """tests/cpu_harness_sens_p.cpp compiled against the problem's generated header (built by build(), else here)."""
    if b.name not in _SENS_P_HARNESS:
        import os
        import __graft_entry__ as entry
        from mpc_code_b200.build import build_dir_for
        res = b.lib
        path = entry.harness_path(res, b.name, entry.SENS_P_HARNESS)
        if not os.path.exists(path):
            d = build_dir_for(os.path.dirname(path), os.path.basename(path))
            os.makedirs(d, exist_ok=True)
            path = os.path.join(d, os.path.basename(path))
            if not os.path.exists(path):
                entry.build_harness(os.path.dirname(res["header"]), path, entry.SENS_P_HARNESS)
        _SENS_P_HARNESS[b.name] = ctypes.CDLL(path)
    return _SENS_P_HARNESS[b.name]


def n_params(p):
    return p.nd + (p.npx + p.npy) * p.N


def par_index(b, j):
    """Index into par of component j of p."""
    off = b.ocp.off
    return off["d"] + j if j < b.prob.nd else off["px"] + (j - b.prob.nd)


def harness_sens_p(b, par, w0, dp=None, gw=None, dtheta=None, theta_only=0, tol=TIGHT, max_iter=200):
    """Solve, factor_p (or only the theta part), JVP_p, VJP_p and the theta JVP / VJP on the same capture."""
    H, p = sens_p_harness(b), b.prob
    par = np.ascontiguousarray(np.atleast_2d(par), dtype=float)
    B, nth, npp = par.shape[0], 2 * (p.nx + p.nu), n_params(p)
    w = np.ascontiguousarray(np.broadcast_to(np.atleast_2d(w0), (B, p.nw)), dtype=float).copy()
    dp = np.zeros((B, 0, npp)) if dp is None else np.ascontiguousarray(dp, dtype=float)
    dtheta = np.zeros((B, 0, nth)) if dtheta is None else np.ascontiguousarray(dtheta, dtype=float)
    gw = np.zeros((B, p.nw)) if gw is None else np.ascontiguousarray(gw, dtype=float)
    f = np.zeros(B); st = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32); sst = np.zeros(B, dtype=np.int32)
    dw = np.zeros((B, dp.shape[1], p.nw)); gp = np.zeros((B, npp))
    dw_th = np.zeros((B, dtheta.shape[1], p.nw)); gth = np.zeros((B, nth))
    H.h_sens_size_p.restype = ctypes.c_long
    H.h_sens_size_theta.restype = ctypes.c_long
    fac = np.zeros(B * max(int(H.h_sens_size_p()), 0))
    lbg, ubg = b.ocp_range_bounds()
    if lbg.size == 0:
        lbg = ubg = np.zeros(1)
    lbx, ubx = np.ascontiguousarray(b.ocp.w_lb), np.ascontiguousarray(b.ocp.w_ub)
    H.h_ocp_sens_p.argtypes = [ctypes.c_int] + [VP] * 9 + [ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                                         ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int] + \
        [VP] * 4 + [ctypes.c_int] + [VP] * 5
    rc = H.h_ocp_sens_p(B, par.ctypes.data, w.ctypes.data, f.ctypes.data, st.ctypes.data, it.ctypes.data,
                        lbx.ctypes.data, ubx.ctypes.data, lbg.ctypes.data, ubg.ctypes.data, max_iter, tol, 0.1, 1e-8, 0,
                        theta_only, dp.shape[1], dp.ctypes.data, dw.ctypes.data, gw.ctypes.data, gp.ctypes.data,
                        dtheta.shape[1], dtheta.ctypes.data, dw_th.ctypes.data, gth.ctypes.data, sst.ctypes.data,
                        fac.ctypes.data if fac.size else None)
    return dict(rc=rc, w=w, status=st, sstatus=sst, dw=dw, gp=gp, dw_th=dw_th, gtheta=gth, fac=fac,
                theta_size=int(H.h_sens_size_theta()))


def unit_dirs(B, n):
    return np.broadcast_to(np.eye(n), (B, n, n)).copy()


_SMODS_P = {}


def anchor_p(b, par, w0, gap=1e-4, tol=TIGHT):
    """Active-set dw/dp [nw, n_p] at the oracle solution and whether its active set is clear."""
    import sensitivity_p_anchor as osens
    from oracle.nlp import OcpNlp
    if b.name not in _SMODS_P:
        _SMODS_P[b.name] = osens.build_p(b.name, b.ocp)
    res, lb, ub = oracle_solve(b, par, w0, tol=tol)
    assert res.status == 0
    nlp = OcpNlp(b.ocp, b.oracle)
    dW, clear = osens.active_set_jacobian_p(nlp, _SMODS_P[b.name], res, par, lb, ub, b.ocp.g_lb, b.ocp.g_ub, gap=gap)
    return dW, clear, res


def _loop_cases(b, steps=7):
    """The OCP parameters and warm starts of steps 1.. of the problem's closed loop run by the device code on the CPU."""
    from harness_loop import HarnessLoop
    seen = []
    solve = b.harness_ocp

    def spy(par, w0, *args, **kwargs):
        seen.append((np.atleast_2d(par).copy(), np.atleast_2d(w0).copy()))
        return solve(par, w0, *args, **kwargs)

    b.harness_ocp = spy
    try:
        HarnessLoop(b, 1).run(steps)
    finally:
        del b.harness_ocp
    return np.concatenate([s[0] for s in seen[1:]]), np.concatenate([s[1] for s in seen[1:]])


def _cases(b):
    if b.name == "nmpc_cstr":
        return G["ocp_par"][:6], G["ocp_w0"]
    if b.name == "nmpc_dis":       # its clamped discrete map leaves the random points of sample_pars infeasible
        return _loop_cases(b)
    return sample_pars(b), b.cold_guess()


# nmpc_dis: the clamps of its discrete map (if_else) stop the solves short of 1e-12
TOL = {"nmpc_dis": 1e-10}


def fd_columns(b):
    """d[1] (inside the RK4 ODE of Ex_NMPC), and a px_k and a py_k component at an early, a middle and a late stage."""
    p = b.prob
    N = p.N
    cols = [1] if p.nd > 1 else [0]
    for k in (0, N // 2, N - 1):
        cols.append(p.nd + k * p.npx + (k % p.npx))
        cols.append(p.nd + p.npx * N + k * p.npy + (k % p.npy))
    return cols


# ---- (1) the p-anchor agrees with finite differences of the oracle -----------------------------------------------------
def test_p_anchor_matches_oracle_finite_differences(nmpc):
    pars, w0 = _cases(nmpc)
    cols = fd_columns(nmpc)
    checked = 0
    for par in pars:
        dW, clear, res = anchor_p(nmpc, par, w0)
        if not clear:
            continue
        fd = np.zeros((dW.shape[0], len(cols)))
        for t, j in enumerate(cols):
            pi = par_index(nmpc, j)
            h = 1e-5 * max(1.0, abs(par[pi]))
            pp, pm = par.copy(), par.copy()
            pp[pi] += h; pm[pi] -= h
            rp, _, _ = oracle_solve(nmpc, pp, res.x)
            rm, _, _ = oracle_solve(nmpc, pm, res.x)
            fd[:, t] = (rp.x - rm.x) / (2 * h)
        assert np.abs(fd[:, [0, 1, 3, 5]]).max(axis=0).min() > 1e-3      # d[1] and the px columns move the solution
        assert np.all(_col_close(fd, dW[:, cols], 1e-5)), np.abs(fd - dW[:, cols]).max(axis=0)
        checked += 1
    assert checked >= 2


# ---- (2) the device arithmetic matches the anchor -------------------------------------------------------------------
PROBLEMS = ["nmpc_cstr", "nmpc_cstr_gineq", "lmpc_wb", "nmpc_dis", "lmpc_cstr_termcons"]
RTOL_ANCHOR = {"lmpc_cstr_termcons": 1e-5}


@pytest.mark.parametrize("name", PROBLEMS)
def test_harness_jvp_p_matches_active_set_anchor(name):
    b = _bundle(name)
    p = b.prob
    npp = n_params(p)
    pars, w0 = _cases(b)
    tol = TOL.get(name, TIGHT)
    r = harness_sens_p(b, pars, w0, unit_dirs(len(pars), npp), tol=tol)
    assert r["rc"] == 0
    checked = 0
    for i, par in enumerate(pars):
        if r["status"][i] != 0:
            continue
        dW, clear, _ = anchor_p(b, par, r["w"][i], gap=1e-3, tol=tol)
        if not clear:
            continue
        assert r["sstatus"][i] == 0
        J = r["dw"][i].T                                       # [nw, n_p]
        assert np.all(J[:p.nx] == 0.0)                         # x_0 = x_hat does not depend on p
        assert np.all(_col_close(J, dW, RTOL_ANCHOR.get(name, 1e-6))), (name, np.abs(J - dW).max(axis=0))
        checked += 1
    assert checked >= 1, name
    assert np.abs(r["dw"]).max() > 1e-3


# ---- (3) an anchor that shares nothing with the oracle: unconstrained linear MPC in closed form -----------------------
def test_jvp_p_of_linear_mpc_is_the_condensed_least_squares_solution(lmpc_cstr):
    """lmpc_cstr with its bounds inactive is an equality-constrained LQ problem: x_{k+1} = A x_k + B u_k + Bd d + px_k,
    cost sum 1/2 |x_k - x_s|_Q^2 + 1/2 |u_k - u_s|_R^2 + 1/2 |x_N - x_s|_P^2 (P the DARE solution).  Condensing the
    states, X = Phi x_0 + Gam U + Psi v with v = [d; px], gives dU/dv = -(Gam' Qb Gam + Rb)^{-1} Gam' Qb Psi exactly;
    py enters only the (inactive) output rows."""
    import scipy.linalg
    b = lmpc_cstr
    p, ns = b.prob, b.prob.ns
    n, m, N, nd = p.nx, p.nu, p.N, p.nd
    A, Bm, Q, R = [np.asarray(ns[k], dtype=float) for k in ("A", "B", "Q", "R")]
    Bd = np.asarray(ns["Bd"], dtype=float)
    P = scipy.linalg.solve_discrete_are(A, Bm, Q, R)
    nv = nd + n * N
    Gam = np.zeros((n * N, m * N)); Psi = np.zeros((n * N, nv))
    for k in range(N):                                        # rows of x_{k+1}
        for j in range(k + 1):
            Ak = np.linalg.matrix_power(A, k - j)
            Gam[n * k:n * (k + 1), m * j:m * (j + 1)] = Ak @ Bm
            Psi[n * k:n * (k + 1), :nd] += Ak @ Bd
            Psi[n * k:n * (k + 1), nd + n * j:nd + n * (j + 1)] = Ak
    Qb = scipy.linalg.block_diag(*([Q] * (N - 1) + [P])); Rb = scipy.linalg.block_diag(*([R] * N))
    dU = -np.linalg.solve(Gam.T @ Qb @ Gam + Rb, Gam.T @ Qb @ Psi)
    dX = Gam @ dU + Psi
    ref = np.zeros((p.nw, n_params(p)))
    for k in range(N):
        ref[(n + m) * k + n:(n + m) * (k + 1), :nv] = dU[m * k:m * (k + 1)]
        ref[(n + m) * (k + 1):(n + m) * (k + 1) + n, :nv] = dX[n * k:n * (k + 1)]
    rng = np.random.default_rng(3)
    pars = np.array([b.ocp_par(0.1 * rng.uniform(-1, 1, n), np.zeros(n), np.zeros(m), 0.01 * rng.uniform(-1, 1, nd),
                               np.zeros(m)) for _ in range(3)])
    r = harness_sens_p(b, pars, np.zeros(p.nw), unit_dirs(len(pars), n_params(p)))
    assert np.all(r["status"] == 0) and np.all(r["sstatus"] == 0)
    for i in range(len(pars)):
        assert np.abs(r["dw"][i].T - ref).max() <= 1e-8 * np.abs(ref).max(), np.abs(r["dw"][i].T - ref).max()


# ---- (4) adjoint consistency -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", PROBLEMS)
def test_vjp_p_is_the_adjoint_of_the_jvp_p(name):
    b = _bundle(name)
    p = b.prob
    pars, w0 = _cases(b)
    rng = np.random.default_rng(11)
    B = len(pars)
    dp = rng.standard_normal((B, 1, n_params(p))); gw = rng.standard_normal((B, p.nw))
    if b.ocp.G is not None:
        # the user rows of nmpc_cstr_gineq read py_k and are strongly active at these points: they enter the condensed
        # system with Sigma ~ 1e13, and the py columns of the two sweeps differ by the rounding of that condensation
        # (~1e-5 relative; d and px agree to 1e-14).  py through range rows is covered by nmpc_cstr's output rows.
        dp[:, :, p.nd + p.npx * p.N:] = 0.0
    tol = TOL.get(name, TIGHT)
    r = harness_sens_p(b, pars, w0, dp, gw, tol=tol)
    ok = r["sstatus"] == 0
    assert ok.sum() >= 1
    lhs = np.einsum("bw,bw->b", gw, r["dw"][:, 0]); rhs = np.einsum("bt,bt->b", r["gp"], dp[:, 0])
    assert np.all(np.abs(lhs - rhs)[ok] <= 1e-10 * np.maximum(np.abs(lhs), np.abs(rhs))[ok])


# ---- (5) the theta part of a p capture is the theta capture ----------------------------------------------------------
@pytest.mark.parametrize("name", ["nmpc_cstr", "lmpc_wb", "lmpc_cstr_termcons"])
def test_theta_part_of_p_capture_is_bitwise_the_theta_capture(name):
    b = _bundle(name)
    p = b.prob
    nth = 2 * (p.nx + p.nu)
    pars, w0 = _cases(b)
    B = len(pars)
    rng = np.random.default_rng(5)
    dth = rng.standard_normal((B, 2, nth)); gw = rng.standard_normal((B, p.nw))
    H = sens_harness(b)
    H.h_sens_size.restype = ctypes.c_long
    size = int(H.h_sens_size())
    # the theta harness (tests/test_ocp_sensitivity.py), keeping its capture
    par = np.ascontiguousarray(pars, dtype=float)
    w = np.ascontiguousarray(np.broadcast_to(w0, (B, p.nw)), dtype=float).copy()
    f = np.zeros(B); st = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32); sst = np.zeros(B, dtype=np.int32)
    dw_th = np.zeros((B, 2, p.nw)); gth = np.zeros((B, nth)); fac_th = np.zeros(B * size)
    lbg, ubg = b.ocp_range_bounds()
    if lbg.size == 0:
        lbg = ubg = np.zeros(1)
    lbx, ubx = np.ascontiguousarray(b.ocp.w_lb), np.ascontiguousarray(b.ocp.w_ub)
    H.h_ocp_sens.argtypes = [ctypes.c_int] + [VP] * 9 + [ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                                       ctypes.c_int, ctypes.c_int] + [VP] * 6
    H.h_ocp_sens(B, par.ctypes.data, w.ctypes.data, f.ctypes.data, st.ctypes.data, it.ctypes.data, lbx.ctypes.data,
                 ubx.ctypes.data, lbg.ctypes.data, ubg.ctypes.data, 200, TIGHT, 0.1, 1e-8, 0, 2, dth.ctypes.data,
                 dw_th.ctypes.data, gw.ctypes.data, gth.ctypes.data, sst.ctypes.data, fac_th.ctypes.data)
    r = harness_sens_p(b, pars, w0, dtheta=dth, gw=gw)
    assert r["theta_size"] == size and np.array_equal(r["w"], w)
    head = r["fac"][:B * size].reshape(B, size).copy()
    assert np.all(head[:, 1] == 1.0)                           # the mark of the p-blocks; the theta factor leaves it 0
    head[:, 1] = 0.0
    assert np.array_equal(head, fac_th.reshape(B, size))
    assert np.array_equal(r["dw_th"], dw_th) and np.array_equal(r["gtheta"], gth)


# ---- (6) refusals and failure statuses -------------------------------------------------------------------------------
def test_contform_problem_refuses_p_and_keeps_theta():
    from test_ocp_sensitivity import harness_sens
    b = _bundle("enmpc_reactor")
    assert b.lib["gen"]["defines"]["MPCB_SENS_P"] == 0
    assert _bundle("nmpc_cstr").lib["gen"]["defines"]["MPCB_SENS_P"] == 1
    p = b.prob
    pars, w0 = _cases(b)
    r = harness_sens_p(b, pars[:2], w0)
    assert r["rc"] < 0
    nth = 2 * (p.nx + p.nu)
    rt = harness_sens(b, pars[:2], w0, unit_dirs(2, nth))
    assert np.any(rt["sstatus"] == 0) and np.all(np.isfinite(rt["dw"][rt["sstatus"] == 0]))
    lib = ctypes.CDLL(b.lib["so"])
    lib.mpcb_last_error.restype = ctypes.c_char_p
    lib.mpcb_create.argtypes = [ctypes.c_int, VP, VP, ctypes.POINTER(VP)]
    lib.mpcb_ocp_sens_factor_p.argtypes = [VP] * 5
    lib.mpcb_ocp_jvp_p.argtypes = [VP, VP, ctypes.c_int, VP, VP, VP]
    lib.mpcb_ocp_vjp_p.argtypes = [VP] * 5
    h = VP()
    created = lib.mpcb_create(1, None, None, ctypes.byref(h)) == 0   # fails without a GPU; the refusal needs no device
    assert lib.mpcb_ocp_sens_factor_p(h, None, None, None, None) < 0
    assert b"d / px / py" in lib.mpcb_last_error(h)
    assert lib.mpcb_ocp_jvp_p(h, None, 1, None, None, None) < 0
    assert lib.mpcb_ocp_vjp_p(h, None, None, None, None) < 0
    if created:
        lib.mpcb_destroy.argtypes = [VP]
        lib.mpcb_destroy(h)


def test_p_sweeps_on_a_theta_only_capture_give_nan(nmpc):
    p = nmpc.prob
    pars, w0 = _cases(nmpc)
    r = harness_sens_p(nmpc, pars[:2], w0, unit_dirs(2, n_params(p))[:, :4], np.ones((2, p.nw)), theta_only=1)
    assert np.all(r["sstatus"] == 0)
    assert np.all(np.isnan(r["dw"])) and np.all(np.isnan(r["gp"]))


def test_infeasible_solve_gives_status_1_and_nan(lmpc_cstr):
    b = lmpc_cstr
    p = b.prob
    par = b.ocp_par(p.x0_m, p.x0_m, p.u0, np.zeros(p.nd))
    r = harness_sens_p(b, par, b.cold_guess(), unit_dirs(1, n_params(p))[:, :5], np.ones((1, p.nw)), tol=1e-8)
    assert r["status"][0] == 2 and r["sstatus"][0] == 1
    assert np.all(np.isnan(r["dw"])) and np.all(np.isnan(r["gp"]))


# ==== on the device ===================================================================================================
def _sampled_p_dirs(p, count=24, seed=0):
    """The unit directions of d and `count` sampled px / py columns."""
    npp = n_params(p)
    rng = np.random.default_rng(seed)
    cols = np.r_[np.arange(p.nd), np.sort(rng.choice(np.arange(p.nd, npp), count, replace=False))]
    return cols, np.eye(npp)[cols]


@pytest.mark.gpu
def test_device_matches_harness_on_ex_nmpc(nmpc):
    import torch
    p = nmpc.prob
    B, nw, npp = 4096, p.nw, n_params(p)
    cols, E = _sampled_p_dirs(p)
    par = _nmpc_batch(B)
    h, solver = _device_solver(nmpc, B)
    assert h.np_params == npp
    sol = solver(x0=G["ocp_w0"], p=par)
    sens = solver.sensitivity(params=True)
    rng = np.random.default_rng(2)
    gw = rng.standard_normal((B, nw))
    dw = sens.jvp_p(torch.as_tensor(E, device=h.device).expand(B, -1, -1)).cpu().numpy()
    gp = sens.vjp_p(gw).cpu().numpy()
    st = solver.stats()["status"].cpu().numpy(); sst = sens.status.cpu().numpy()
    idx = np.arange(0, B, B // 64)
    r = harness_sens_p(nmpc, par[idx], G["ocp_w0"], np.broadcast_to(E, (len(idx),) + E.shape).copy(), gw[idx],
                       tol=1e-8, max_iter=100)
    assert np.array_equal(r["status"], st[idx]) and np.array_equal(r["sstatus"], sst[idx])
    ok = r["sstatus"] == 0
    assert ok.sum() >= 32
    assert np.abs(sol["x"].cpu().numpy()[idx] - r["w"]).max() < 1e-9
    for j in np.where(ok)[0]:
        assert np.all(_col_close(dw[idx[j]].T, r["dw"][j].T, 1e-9)), np.abs(dw[idx[j]] - r["dw"][j]).max()
        assert np.allclose(gp[idx[j]], r["gp"][j], rtol=1e-9, atol=1e-9 * np.abs(r["gp"][j]).max())
    assert np.all(np.isnan(dw[sst != 0])) and np.all(~np.isnan(dw[sst == 0]))
    # the theta methods accept the p capture
    fac_t, _ = h.ocp_sens_factor(h.tensor(par, p.npar))
    eye = torch.eye(10, dtype=torch.float64, device=h.device).expand(B, -1, -1)
    assert torch.equal(h.ocp_jvp(fac_t, eye), sens.jvp(eye))
    K = sens.disturbance_gain()
    assert K.shape == (B, p.nu, p.nd)
    assert torch.equal(K, sens.jvp_p(torch.eye(npp, dtype=torch.float64, device=h.device)[:p.nd].expand(B, -1, -1))
                       [:, :, p.nx:p.nx + p.nu].transpose(1, 2))


@pytest.mark.gpu
def test_device_jvp_p_matches_device_finite_differences(nmpc):
    from test_ocp_sensitivity import anchor
    p = nmpc.prob
    pars, w0 = G["ocp_par"][:6], G["ocp_w0"]
    clear = np.array([anchor(nmpc, par, w0)[1] for par in pars])
    assert clear.sum() >= 2
    pars = pars[clear]
    nb = len(pars)
    cols = [1, p.nd + (p.N // 2) * p.npx]                         # d[1] and a px_k component
    idx = [par_index(nmpc, j) for j in cols]
    steps = 1e-5 * np.maximum(1.0, np.abs(pars[:, idx]))
    rows = [pars]
    for sgn in (1, -1):
        for t, pi in enumerate(idx):
            q = pars.copy(); q[:, pi] += sgn * steps[:, t]; rows.append(q)
    allp = np.concatenate(rows)
    h, solver = _device_solver(nmpc, allp.shape[0], tol=TIGHT, max_iter=200)
    w = solver(x0=w0, p=allp)["x"].cpu().numpy()
    assert np.all(solver.stats()["status"].cpu().numpy() == 0)
    E = np.eye(n_params(p))[cols]
    dW = solver.sensitivity(params=True).jvp_p(np.broadcast_to(E, (allp.shape[0],) + E.shape).copy()).cpu().numpy()
    nc = len(cols)
    for i in range(nb):
        fd = np.stack([(w[nb * (1 + t) + i] - w[nb * (1 + nc + t) + i]) / (2 * steps[i, t]) for t in range(nc)], axis=1)
        assert np.all(_col_close(dW[i].T, fd, 1e-5)), np.abs(dW[i].T - fd).max(axis=0)


@pytest.mark.gpu
def test_p_capture_is_independent_of_later_solves(nmpc):
    import torch
    p = nmpc.prob
    B = 256
    par1, par2 = _nmpc_batch(B, 1), _nmpc_batch(B, 2)
    rng = np.random.default_rng(4)
    dp = torch.as_tensor(rng.standard_normal((B, 3, n_params(p))), device="cuda")
    gw = torch.as_tensor(rng.standard_normal((B, p.nw)), device="cuda")
    h, solver = _device_solver(nmpc, B)
    solver(x0=G["ocp_w0"], p=par1)
    sens = solver.sensitivity(params=True)
    j1, v1 = sens.jvp_p(dp).clone(), sens.vjp_p(gw).clone()
    out_a = solver(x0=G["ocp_w0"], p=par2)
    st_a = solver.stats()
    st_a = (st_a["status"].clone(), st_a["iter_count"].clone())
    assert torch.equal(sens.jvp_p(dp), j1) and torch.equal(sens.vjp_p(gw), v1)
    # solve -> factor_p -> solve gives the output of solve -> solve, bit for bit
    h2, solver2 = _device_solver(nmpc, B)
    solver2(x0=G["ocp_w0"], p=par1)
    out_b = solver2(x0=G["ocp_w0"], p=par2)
    assert torch.equal(out_a["x"], out_b["x"]) and torch.equal(out_a["f"], out_b["f"])
    assert torch.equal(st_a[0], solver2.stats()["status"]) and torch.equal(st_a[1], solver2.stats()["iter_count"])
    with pytest.raises(RuntimeError, match="params=True"):
        solver2.sensitivity().jvp_p(dp)


@pytest.mark.gpu
def test_ocp_layer_gradient_in_p_matches_finite_differences(nmpc):
    import torch
    from mpc_code_b200.sensitivity import OcpLayer, params_of, theta_of
    p = nmpc.prob
    pars = torch.as_tensor(G["ocp_par"][:4], device="cuda")
    h, solver = _device_solver(nmpc, 4, tol=TIGHT, max_iter=200)
    layer = OcpLayer(solver, params=True)
    w0 = torch.as_tensor(G["ocp_w0"], device="cuda").expand(4, -1).contiguous()
    theta = theta_of(pars, p.nx, p.nu, p.nd).clone().requires_grad_(True)
    pp = params_of(pars, p.nx, p.nu, p.nd, p.ny).clone().requires_grad_(True)

    def loss_of(th, q):
        w = layer(th, pars, w0, q)
        return (w[:, p.nx:p.nx + p.nu] ** 2).sum(dim=1)

    loss = loss_of(theta, pp)
    ok = (solver.stats()["status"] == 0) & (layer.last.status == 0)
    assert bool(ok.any())
    loss.sum().backward()
    g = pp.grad.cpu().numpy()
    cols = fd_columns(nmpc)
    fd = np.zeros((4, len(cols)))
    with torch.no_grad():
        for t, j in enumerate(cols):
            e = torch.zeros_like(pp); e[:, j] = 1.0
            hstep = 1e-5 * torch.clamp(pp.abs()[:, j:j + 1], min=1.0)
            fd[:, t] = ((loss_of(theta, pp + hstep * e) - loss_of(theta, pp - hstep * e)) / (2 * hstep[:, 0])).cpu().numpy()
    for i in np.where(ok.cpu().numpy())[0]:
        assert np.allclose(g[i, cols], fd[i], rtol=1e-5, atol=1e-5 * np.abs(fd[i]).max()), (g[i, cols], fd[i])
    assert theta.grad is not None and bool(torch.isfinite(theta.grad[ok]).all())
    with pytest.raises(ValueError):
        layer(theta, pars.clone().requires_grad_(True), w0, pp)
    with pytest.raises(ValueError):
        OcpLayer(solver)(theta, pars, w0, pp)
