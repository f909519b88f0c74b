"""Sensitivities of the batched OCP solution (csrc/mpcb_sens.cuh, mpcb_ocp_sens_factor / mpcb_ocp_jvp / mpcb_ocp_vjp).

Without a GPU the device arithmetic runs on the CPU through tests/cpu_harness.cpp and is checked against the
active-set anchor of oracle/sensitivity.py, finite differences of the oracle solve, adjoint consistency and the DARE
gain of a linear MPC.  The `-m gpu` tests repeat the comparisons through the C ABI and the Python layer on the device.
"""
import ctypes
import os

import numpy as np
import pytest

from conftest import GOLDEN, _bundle

VP = ctypes.c_void_p
G = np.load(os.path.join(GOLDEN, "nmpc_oracle.npz"))
TIGHT = 1e-12


def theta_index(p):
    nx, nu, nd = p.nx, p.nu, p.nd
    return np.r_[np.arange(2 * nx + nu), 2 * nx + nu + nd + np.arange(nu)]


_SENS_HARNESS = {}


def sens_harness(b):
    """tests/cpu_harness_sens.cpp compiled against the problem's generated header (built by build(), else here)."""
    if b.name not in _SENS_HARNESS:
        import __graft_entry__ as entry
        from mpc_code_b200.build import build_dir_for
        res = b.lib
        path = entry.harness_path(res, b.name, entry.SENS_HARNESS)
        if not os.path.exists(path):
            d = build_dir_for(os.path.dirname(path), os.path.basename(path))
            os.makedirs(d, exist_ok=True)
            path = os.path.join(d, os.path.basename(path))
            if not os.path.exists(path):
                entry.build_harness(os.path.dirname(res["header"]), path, entry.SENS_HARNESS)
        _SENS_HARNESS[b.name] = ctypes.CDLL(path)
    return _SENS_HARNESS[b.name]


def harness_sens(b, par, w0, dtheta=None, gw=None, tol=TIGHT, max_iter=200):
    """Solve, factor, JVP and VJP in one harness call.  dtheta [B, ndir, ntheta], gw [B, nw]."""
    H, p = sens_harness(b), b.prob
    par = np.ascontiguousarray(np.atleast_2d(par), dtype=float)
    B, nth = par.shape[0], 2 * (p.nx + p.nu)
    w = np.ascontiguousarray(np.broadcast_to(np.atleast_2d(w0), (B, p.nw)), dtype=float).copy()
    dtheta = np.zeros((B, 0, nth)) if dtheta is None else np.ascontiguousarray(dtheta, dtype=float)
    gw = np.zeros((B, p.nw)) if gw is None else np.ascontiguousarray(gw, dtype=float)
    ndir = dtheta.shape[1]
    f = np.zeros(B); st = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32); sst = np.zeros(B, dtype=np.int32)
    dw = np.zeros((B, ndir, p.nw)); gth = np.zeros((B, nth))
    lbg, ubg = b.ocp_range_bounds()
    if lbg.size == 0:
        lbg = ubg = np.zeros(1)
    lbx, ubx = np.ascontiguousarray(b.ocp.w_lb), np.ascontiguousarray(b.ocp.w_ub)
    H.h_ocp_sens.argtypes = [ctypes.c_int] + [VP] * 9 + [ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                                       ctypes.c_int, ctypes.c_int] + [VP] * 6
    H.h_ocp_sens(B, par.ctypes.data, w.ctypes.data, f.ctypes.data, st.ctypes.data, it.ctypes.data, lbx.ctypes.data,
                 ubx.ctypes.data, lbg.ctypes.data, ubg.ctypes.data, max_iter, tol, 0.1, 1e-8, 0, ndir, dtheta.ctypes.data,
                 dw.ctypes.data, gw.ctypes.data, gth.ctypes.data, sst.ctypes.data, None)
    return dict(w=w, status=st, sstatus=sst, dw=dw, gtheta=gth)


def unit_dirs(B, nth):
    return np.broadcast_to(np.eye(nth), (B, nth, nth)).copy()


def oracle_solve(b, par, w0, tol=TIGHT):
    from oracle.ipm import IpmOptions
    from oracle.nlp import OcpNlp
    n = b.prob.nx
    lb, ub = b.ocp.w_lb.copy(), b.ocp.w_ub.copy()
    lb[:n] = ub[:n] = par[:n]
    return OcpNlp(b.ocp, b.oracle).solve(w0, par, lb, ub, opts=IpmOptions(max_iter=200, tol=tol)), lb, ub


_SMODS = {}


def anchor(b, par, w0, gap=1e-4):
    """Active-set dw/dtheta [nw, ntheta] at the oracle solution and whether its active set is clear (inactive bounds at
    a distance > gap)."""
    from oracle import sensitivity as osens
    from oracle.nlp import OcpNlp
    if b.name not in _SMODS:
        _SMODS[b.name] = osens.build(b.name, b.ocp)
    res, lb, ub = oracle_solve(b, par, w0)
    assert res.status == 0
    nlp = OcpNlp(b.ocp, b.oracle)
    dW, clear = osens.active_set_jacobian(nlp, _SMODS[b.name], res, par, lb, ub, b.ocp.g_lb, b.ocp.g_ub, gap=gap)
    return dW, clear, res


def sample_pars(b, count=6, seed=0):
    """Parameter vectors around the problem's nominal point: perturbed estimate, targets near the initial state."""
    p = b.prob
    rng = np.random.default_rng(seed)
    d = np.asarray(p.dhat0, dtype=float) if p.nd else np.zeros(0)
    out = []
    for _ in range(count):
        xhat = p.x0_m * (1 + 0.01 * rng.uniform(-1, 1, p.nx))
        xs = p.x0_m * (1 + 0.01 * rng.uniform(-1, 1, p.nx))
        us = p.u0 * (1 + 0.01 * rng.uniform(-1, 1, p.nu))
        um1 = p.u0 * (1 + 0.01 * rng.uniform(-1, 1, p.nu))
        out.append(b.ocp_par(xhat, xs, us, d, um1))
    return np.array(out)


def _cases(b):
    if b.name == "nmpc_cstr":
        return G["ocp_par"][:6], G["ocp_w0"]
    return sample_pars(b), b.cold_guess()


def _col_close(A, R, rtol):
    """Column-wise: |A - R| <= rtol * max(|R| of the column, 1e-3 max|R|)."""
    scale = np.maximum(np.abs(R).max(axis=0), 1e-3 * max(np.abs(R).max(), 1e-300))
    return np.abs(A - R).max(axis=0) <= rtol * scale


# ---- (1) the anchor agrees with finite differences of the oracle ------------------------------------------------------
def test_active_set_anchor_matches_oracle_finite_differences(nmpc):
    p = nmpc.prob
    idx = theta_index(p)
    pars, w0 = _cases(nmpc)
    checked = 0
    for par in pars:
        dW, clear, res = anchor(nmpc, par, w0)
        if not clear:
            continue
        fd = np.zeros_like(dW)
        for t, pi in enumerate(idx):
            h = 1e-5 * max(1.0, abs(par[pi]))
            pp, pm = par.copy(), par.copy()
            pp[pi] += h; pm[pi] -= h
            rp, _, _ = oracle_solve(nmpc, pp, res.x)
            rm, _, _ = oracle_solve(nmpc, pm, res.x)
            fd[:, t] = (rp.x - rm.x) / (2 * h)
        assert np.all(_col_close(fd, dW, 1e-5)), np.abs(fd - dW).max(axis=0)
        checked += 1
    assert checked >= 2


# ---- (2) the device arithmetic matches the anchor -------------------------------------------------------------------
PROBLEMS = ["nmpc_cstr", "nmpc_cstr_termcons", "nmpc_cstr_gineq", "lmpc_wb", "enmpc_reactor"]
# With the terminal equality the x_s columns reach |dw/dx_s| ~ 360 through the inverse of a poorly conditioned
# reachability Gramian, and the strongly active bounds enter the condensed system with Sigma ~ z^2/mu ~ 1e13: the
# rounding of that condensation shows at ~2e-6 of the column (one instance of six); the anchor eliminates them exactly.
RTOL_ANCHOR = {"nmpc_cstr_termcons": 1e-5}


@pytest.mark.parametrize("name", PROBLEMS)
def test_harness_jvp_matches_active_set_anchor(name):
    b = _bundle(name)
    p = b.prob
    nth = 2 * (p.nx + p.nu)
    pars, w0 = _cases(b)
    r = harness_sens(b, pars, w0, unit_dirs(len(pars), nth))
    checked = 0
    for i, par in enumerate(pars):
        if r["status"][i] != 0:
            continue
        # the device derivative is the barrier system's at the final mu (~1e-13): an inactive bound at distance d adds
        # Sigma ~ mu / d^2 to the Hessian, so the 1e-6 comparison uses instances whose inactive bounds are 1e-3 away
        dW, clear, _ = anchor(b, par, r["w"][i], gap=1e-3)
        if not clear:
            continue
        assert r["sstatus"][i] == 0
        J = r["dw"][i].T                                      # [nw, ntheta]
        assert np.array_equal(J[:p.nx, :p.nx], np.eye(p.nx))  # x_0 is eliminated: dw[0:nx] = dx_hat exactly
        assert np.all(_col_close(J, dW, RTOL_ANCHOR.get(name, 1e-6))), (name, np.abs(J - dW).max(axis=0))
        checked += 1
    assert checked >= 1, name
    if p.nu and b.ocp.uses_uprev:                             # Delta-u form: the u_{k-1} columns are not trivial
        assert np.abs(r["dw"][:, nth - p.nu:, p.nx:p.nx + p.nu]).max() > 1e-3


# ---- (3) LQR gain ----------------------------------------------------------------------------------------------------
def test_feedback_gain_of_linear_mpc_is_the_dare_gain(lmpc_cstr):
    """The terminal weight of lmpc_cstr is the DARE solution, so the finite-horizon Riccati recursion is stationary and
    the gain of an unconstrained solve is the LQR gain (P from SciPy, not from the package)."""
    import scipy.linalg
    b = lmpc_cstr
    p, ns = b.prob, b.prob.ns
    n, m = p.nx, p.nu
    A, Bm, Q, R = [np.asarray(ns[k], dtype=float) for k in ("A", "B", "Q", "R")]
    P = scipy.linalg.solve_discrete_are(A, Bm, Q, R)
    K = -np.linalg.solve(R + Bm.T @ P @ Bm, Bm.T @ P @ A)
    rng = np.random.default_rng(3)
    pars = np.array([b.ocp_par(0.1 * rng.uniform(-1, 1, n), np.zeros(n), np.zeros(m), np.zeros(p.nd), np.zeros(m))
                     for _ in range(4)])
    nth = 2 * (n + m)
    r = harness_sens(b, pars, np.zeros(p.nw), unit_dirs(len(pars), nth))
    assert np.all(r["status"] == 0) and np.all(r["sstatus"] == 0)
    gain = r["dw"][:, :n, n:n + m].transpose(0, 2, 1)         # [B, nu, nx] = dU_0 / dx_hat
    assert np.allclose(gain, K[None], rtol=1e-6, atol=1e-6 * np.abs(K).max()), np.abs(gain - K).max()


# ---- (4) adjoint consistency -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", PROBLEMS)
def test_vjp_is_the_adjoint_of_the_jvp(name):
    b = _bundle(name)
    p = b.prob
    nth = 2 * (p.nx + p.nu)
    pars, w0 = _cases(b)
    rng = np.random.default_rng(11)
    B = len(pars)
    dth = rng.standard_normal((B, 1, nth)); gw = rng.standard_normal((B, p.nw))
    r = harness_sens(b, pars, w0, dth, gw)
    ok = r["sstatus"] == 0
    assert ok.sum() >= 1
    lhs = np.einsum("bw,bw->b", gw, r["dw"][:, 0]); rhs = np.einsum("bt,bt->b", r["gtheta"], dth[:, 0])
    assert np.all(np.abs(lhs - rhs)[ok] <= 1e-10 * np.maximum(np.abs(lhs), np.abs(rhs))[ok])


# ---- (5) failure statuses --------------------------------------------------------------------------------------------
def test_infeasible_solve_gives_status_1_and_nan(lmpc_cstr):
    b = lmpc_cstr
    p = b.prob
    nth = 2 * (p.nx + p.nu)
    par = b.ocp_par(p.x0_m, p.x0_m, p.u0, np.zeros(p.nd))
    r = harness_sens(b, par, b.cold_guess(), unit_dirs(1, nth), np.ones((1, p.nw)), tol=1e-8)
    assert r["status"][0] == 2 and r["sstatus"][0] == 1
    assert np.all(np.isnan(r["dw"])) and np.all(np.isnan(r["gtheta"]))


def test_contform_integrand_depending_on_targets_is_refused():
    """No shipped example integrates a cost that depends on the targets: enmpc_reactor with a u_s term added."""
    import __graft_entry__ as entry
    from mpc_code_b200.build import build_library
    from mpc_code_b200.loader import load_example
    from mpc_code_b200.problem import build_problem, make_specs
    ns = load_example(entry.EXAMPLES["enmpc_reactor"])
    f0 = ns["User_fobj_Cont"]
    ns["User_fobj_Cont"] = lambda x, u, y, xs, us, ys: f0(x, u, y, xs, us, ys) + 1e-3 * (u[0] - us[0]) ** 2
    prob = build_problem(ns)
    ss, ocp = make_specs(prob)
    res = build_library("enmpc_reactor_us", prob, ss, ocp)
    assert res["gen"]["defines"]["MPCB_SENS_CONT_DEP"] == 1
    assert _bundle("enmpc_reactor").lib["gen"]["defines"]["MPCB_SENS_CONT_DEP"] == 0
    lib = ctypes.CDLL(res["so"])
    lib.mpcb_last_error.restype = ctypes.c_char_p
    lib.mpcb_create.argtypes = [ctypes.c_int, VP, VP, ctypes.POINTER(VP)]
    lib.mpcb_ocp_jvp.argtypes = [VP, VP, ctypes.c_int, VP, VP, VP]
    lib.mpcb_ocp_vjp.argtypes = [VP] * 5
    h = VP()
    created = lib.mpcb_create(1, None, None, ctypes.byref(h)) == 0   # fails without a GPU; the refusal needs no device
    assert lib.mpcb_ocp_jvp(h, None, 1, None, None, None) < 0
    assert b"ContForm" in lib.mpcb_last_error(h)
    assert lib.mpcb_ocp_vjp(h, None, None, None, None) < 0
    if created:
        lib.mpcb_destroy.argtypes = [VP]
        lib.mpcb_destroy(h)


# ==== on the device ===================================================================================================
def _device_solver(b, batch, **opts):
    from mpc_code_b200.solvers import BatchedNlpSolver, MpcbHandle, MpcbLibrary
    h = MpcbHandle(MpcbLibrary(b.lib["so"]), batch, opts_dyn=opts or None)
    return h, BatchedNlpSolver("ocp", b.ocp).attach(h)


def _nmpc_batch(B, seed=0):
    """B parameter vectors of Ex_NMPC: the golden OCP instances with perturbed estimates and targets."""
    p = _bundle("nmpc_cstr").prob
    rng = np.random.default_rng(seed)
    par = G["ocp_par"][np.arange(B) % G["ocp_par"].shape[0]].copy()
    par[:, :2 * p.nx] *= 1 + 0.002 * rng.uniform(-1, 1, (B, 2 * p.nx))
    return par


@pytest.mark.gpu
def test_device_matches_harness_on_ex_nmpc(nmpc):
    import torch
    B, nth, nw = 4096, 10, nmpc.prob.nw
    par = _nmpc_batch(B)
    h, solver = _device_solver(nmpc, B)
    sol = solver(x0=G["ocp_w0"], p=par)
    sens = solver.sensitivity()
    rng = np.random.default_rng(2)
    gw = rng.standard_normal((B, nw))
    dw = sens.jvp(torch.eye(nth, dtype=torch.float64, device=h.device).expand(B, -1, -1)).cpu().numpy()
    gth = sens.vjp(gw).cpu().numpy()
    st = solver.stats()["status"].cpu().numpy(); sst = sens.status.cpu().numpy()
    idx = np.arange(0, B, B // 64)
    r = harness_sens(nmpc, par[idx], G["ocp_w0"], unit_dirs(len(idx), nth), gw[idx], tol=1e-8, max_iter=100)
    assert np.array_equal(r["status"], st[idx]) and np.array_equal(r["sstatus"], sst[idx])
    ok = r["sstatus"] == 0
    assert ok.sum() >= 32
    assert np.abs(sol["x"].cpu().numpy()[idx] - r["w"]).max() < 1e-9
    for j in np.where(ok)[0]:
        assert np.all(_col_close(dw[idx[j]].T, r["dw"][j].T, 1e-9)), np.abs(dw[idx[j]] - r["dw"][j]).max()
        assert np.allclose(gth[idx[j]], r["gtheta"][j], rtol=1e-9, atol=1e-9 * np.abs(r["gtheta"][j]).max())
    assert np.all(np.isnan(dw[sst != 0])) and np.all(~np.isnan(dw[sst == 0]))


@pytest.mark.gpu
def test_device_jvp_matches_device_finite_differences(nmpc):
    pars, w0 = G["ocp_par"][:6], G["ocp_w0"]
    clear = np.array([anchor(nmpc, par, w0)[1] for par in pars])
    assert clear.sum() >= 2
    pars = pars[clear]
    nb, nth = len(pars), 10
    idx = theta_index(nmpc.prob)
    steps = 1e-5 * np.maximum(1.0, np.abs(pars[:, idx]))
    rows = [pars]
    for sgn in (1, -1):
        for t, pi in enumerate(idx):
            q = pars.copy(); q[:, pi] += sgn * steps[:, t]; rows.append(q)
    allp = np.concatenate(rows)
    h, solver = _device_solver(nmpc, allp.shape[0], tol=TIGHT, max_iter=200)
    w = solver(x0=w0, p=allp)["x"].cpu().numpy()
    assert np.all(solver.stats()["status"].cpu().numpy() == 0)
    dW = solver.sensitivity().jvp(np.broadcast_to(np.eye(nth), (allp.shape[0], nth, nth)).copy()).cpu().numpy()
    for i in range(nb):
        fd = np.stack([(w[nb * (1 + t) + i] - w[nb * (1 + nth + t) + i]) / (2 * steps[i, t]) for t in range(nth)], axis=1)
        assert np.all(_col_close(dW[i].T, fd, 1e-5)), np.abs(dW[i].T - fd).max(axis=0)


@pytest.mark.gpu
def test_capture_is_independent_of_later_solves(nmpc):
    import torch
    B, nth = 256, 10
    par1, par2 = _nmpc_batch(B, 1), _nmpc_batch(B, 2)
    rng = np.random.default_rng(4)
    dth = torch.as_tensor(rng.standard_normal((B, 3, nth)), device="cuda")
    gw = torch.as_tensor(rng.standard_normal((B, nmpc.prob.nw)), device="cuda")
    h, solver = _device_solver(nmpc, B)
    solver(x0=G["ocp_w0"], p=par1)
    sens = solver.sensitivity()
    j1, v1 = sens.jvp(dth).clone(), sens.vjp(gw).clone()
    out_a = solver(x0=G["ocp_w0"], p=par2)                     # a later solve on the same handle
    st_a = solver.stats()
    st_a = (st_a["status"].clone(), st_a["iter_count"].clone())
    assert torch.equal(sens.jvp(dth), j1) and torch.equal(sens.vjp(gw), v1)
    # solve -> factor -> solve gives the output of solve -> solve, bit for bit
    h2, solver2 = _device_solver(nmpc, B)
    solver2(x0=G["ocp_w0"], p=par1)
    out_b = solver2(x0=G["ocp_w0"], p=par2)
    assert torch.equal(out_a["x"], out_b["x"]) and torch.equal(out_a["f"], out_b["f"])
    assert torch.equal(st_a[0], solver2.stats()["status"]) and torch.equal(st_a[1], solver2.stats()["iter_count"])
    # a solve that bypasses the solver object makes its record stale
    solver.handle.ocp(par1, G["ocp_w0"])
    with pytest.raises(RuntimeError, match="solved another OCP"):
        solver.sensitivity()


@pytest.mark.gpu
def test_ocp_layer_gradient_matches_finite_differences(nmpc):
    import torch
    from mpc_code_b200.sensitivity import OcpLayer, theta_of
    p = nmpc.prob
    pars = torch.as_tensor(G["ocp_par"][:4], device="cuda")
    h, solver = _device_solver(nmpc, 4, tol=TIGHT, max_iter=200)
    layer = OcpLayer(solver)
    w0 = torch.as_tensor(G["ocp_w0"], device="cuda").expand(4, -1).contiguous()
    theta = theta_of(pars, p.nx, p.nu, p.nd).clone().requires_grad_(True)

    def loss_of(th):
        w = layer(th, pars, w0)
        return (w[:, p.nx:p.nx + p.nu] ** 2).sum(dim=1)            # sum of U_0^2, per instance

    loss = loss_of(theta)
    ok = (solver.stats()["status"] == 0) & (layer.last.status == 0)
    assert bool(ok.any())
    loss.sum().backward()
    g = theta.grad.cpu().numpy()
    fd = np.zeros_like(g)
    with torch.no_grad():
        for t in range(theta.shape[1]):
            e = torch.zeros_like(theta); e[:, t] = 1.0
            hstep = 1e-5 * torch.clamp(theta.abs()[:, t:t + 1], min=1.0)
            fd[:, t] = ((loss_of(theta + hstep * e) - loss_of(theta - hstep * e)) / (2 * hstep[:, 0])).cpu().numpy()
    for i in np.where(ok.cpu().numpy())[0]:
        assert np.allclose(g[i], fd[i], rtol=1e-5, atol=1e-5 * np.abs(fd[i]).max()), (g[i], fd[i])
    with pytest.raises(ValueError):
        layer(theta, pars.clone().requires_grad_(True), w0)
    with pytest.raises(ValueError):
        layer(theta, pars, w0.clone().requires_grad_(True))


@pytest.mark.gpu
def test_controller_feedback_gain(nmpc):
    import torch
    from mpc_code_b200.mpc_loop import CompiledProblem
    cp = CompiledProblem(nmpc.prob, "nmpc_cstr")
    ctl = cp.controller(16)
    ctl.step()
    ctl.step()
    K = ctl.feedback_gain()
    K2 = ctl.solver.sensitivity().feedback_gain()
    assert K.shape == (16, nmpc.prob.nu, nmpc.prob.nx) and torch.equal(K, K2)
    assert bool(torch.isfinite(K[ctl.solver.stats()["status"] == 0]).all())
    ctl2 = cp.controller(4)
    ctl2.step_fused()
    with pytest.raises(RuntimeError, match="step_fused"):
        ctl2.feedback_gain()
    with pytest.raises(NotImplementedError):
        ctl2.solver_ss.sensitivity()
