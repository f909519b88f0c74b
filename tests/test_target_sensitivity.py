"""Sensitivities of the steady-state target solution with respect to theta_ss = [usp | ysp | xsp | d | Us_prev | px | py]
(csrc/mpcb_target.cuh, mpcb_target_sens_factor / mpcb_target_jvp / mpcb_target_vjp), and the controller's total gains
through the target problem (BatchedMpc.controller_gains).

Without a GPU the device arithmetic runs on the CPU through tests/cpu_harness_sens_tgt.cpp and is checked against the
active-set anchor of tests/target_sens_anchor.py (itself checked against finite differences of the oracle's target
solve), against the KKT solution of lmpc_cstr's equality-constrained QP in NumPy, for adjoint consistency, and, composed
with the OCP harnesses, against finite differences of the oracle's target + OCP chain.  The `-m gpu` tests repeat the
comparisons through the C ABI and the Python layer on the device.
"""
import ctypes
import os

import numpy as np
import pytest

from conftest import _bundle
from test_ocp_sensitivity import G, TIGHT, _col_close, harness_sens, oracle_solve, unit_dirs
from test_ocp_sensitivity_params import harness_sens_p

VP = ctypes.c_void_p
_HARNESS = {}
_SMODS = {}


def tgt_harness(b):
    """tests/cpu_harness_sens_tgt.cpp compiled against the problem's generated header (built by build(), else here)."""
    if b.name not in _HARNESS:
        import __graft_entry__ as entry
        from mpc_code_b200.build import build_dir_for
        res = b.lib
        path = entry.harness_path(res, b.name, entry.SENS_TGT_HARNESS)
        if not os.path.exists(path):
            d = build_dir_for(os.path.dirname(path), os.path.basename(path))
            os.makedirs(d, exist_ok=True)
            path = os.path.join(d, os.path.basename(path))
            if not os.path.exists(path):
                entry.build_harness(os.path.dirname(res["header"]), path, entry.SENS_TGT_HARNESS)
        _HARNESS[b.name] = ctypes.CDLL(path)
    return _HARNESS[b.name]


def n_theta_ss(p):
    return 2 * p.nu + p.ny + p.nx + p.nd + p.npx + p.npy


def harness_tgt(b, par, w0, dth=None, gw=None, lbx=None, ubx=None, tol=TIGHT, max_iter=200, fac=False, mu_init=0.1,
                relax=1e-8, honor=0):
    """Solve, capture, JVP and VJP of the target problem on the CPU."""
    H, p, ss = tgt_harness(b), b.prob, b.ss
    par = np.ascontiguousarray(np.atleast_2d(par), dtype=float)
    B, nth = par.shape[0], n_theta_ss(p)
    w0 = np.ascontiguousarray(np.broadcast_to(np.atleast_2d(w0), (B, ss.nw)), dtype=float)
    dth = np.zeros((B, 0, nth)) if dth is None else np.ascontiguousarray(dth, dtype=float)
    gw = np.zeros((B, ss.nw)) if gw is None else np.ascontiguousarray(gw, dtype=float)
    lbx = np.ascontiguousarray(ss.w_lb if lbx is None else lbx, dtype=float)
    ubx = np.ascontiguousarray(ss.w_ub if ubx is None else ubx, dtype=float)
    w = np.zeros((B, ss.nw)); st = np.zeros(B, dtype=np.int32); sst = np.zeros(B, dtype=np.int32)
    dw = np.zeros((B, dth.shape[1], ss.nw)); gth = np.zeros((B, nth))
    H.h_tgt_sens_size.restype = ctypes.c_long
    cap = np.zeros(B * max(int(H.h_tgt_sens_size()), 0)) if fac else None
    H.h_target_sens.argtypes = [ctypes.c_int] + [VP] * 7 + [ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                                             ctypes.c_double, ctypes.c_int, ctypes.c_int] + [VP] * 5
    rc = H.h_target_sens(B, par.ctypes.data, w0.ctypes.data, w.ctypes.data, st.ctypes.data, sst.ctypes.data,
                         lbx.ctypes.data, ubx.ctypes.data, max_iter, tol, mu_init, relax, honor, dth.shape[1], dth.ctypes.data,
                         dw.ctypes.data, gw.ctypes.data, gth.ctypes.data, cap.ctypes.data if cap is not None else None)
    assert rc == 0
    return dict(w=w, status=st, sstatus=sst, dw=dw, gth=gth, fac=cap)


def target_par(b, rng=None, scale=1.0):
    """par_ss of the problem's nominal point (set-points at t = 0, d = dhat0, Us_prev = u0, lam = 0), randomly perturbed
    (with a small lam, through which Us_prev reaches the output rows)."""
    p, ss = b.prob, b.ss
    off = ss.off
    par = np.zeros(ss.npar)
    if p.defSP is not None:
        ysp, usp, xsp = [np.asarray(v, dtype=float).ravel() for v in p.defSP(0.0)]
    else:
        ysp, usp, xsp = np.zeros(p.ny), np.zeros(p.nu), np.zeros(p.nx)
    d = np.asarray(p.dhat0, dtype=float).ravel() if p.nd else np.zeros(0)
    usprev = np.asarray(p.u0, dtype=float).ravel()
    if rng is not None:
        def wiggle(v):
            return v * (1 + 0.02 * scale * rng.uniform(-1, 1, v.size)) + 0.01 * scale * rng.uniform(-1, 1, v.size)
        ysp, usp, xsp, d, usprev = [wiggle(v) for v in (ysp, usp, xsp, d, usprev)]
    for name, v in (("usp", usp), ("ysp", ysp), ("xsp", xsp), ("d", d), ("usprev", usprev)):
        par[off[name]:off[name] + v.size] = v
    if rng is not None:
        par[off["lam"]:off["lam"] + p.ny * p.nu] = 0.02 * scale * rng.uniform(-1, 1, p.ny * p.nu)
    return par


def target_guess(b, par):
    """The loop's initial guess [x0_m, u0, Fy(x0_m, u0, d)] (MPC_code.py:696-700)."""
    p, off = b.prob, b.ss.off
    d = par[off["d"]:off["d"] + p.nd]
    y0 = b.oracle.orc_fy(p.x0_m, p.u0, d if p.nd else np.zeros(1), np.zeros(1), np.zeros(max(p.npy, 1)))
    return np.concatenate([p.x0_m, p.u0, np.asarray(y0, dtype=float).ravel()])


def oracle_target(b, par, w0, tol=TIGHT):
    from oracle.ipm import IpmOptions
    from oracle.nlp import TargetNlp
    return TargetNlp(b.ss, b.oracle).solve(w0, par, opts=IpmOptions(max_iter=200, tol=tol))


def anchor(b, par, w0, gap=1e-4):
    import target_sens_anchor as tsa
    from oracle.nlp import TargetNlp
    if b.name not in _SMODS:
        _SMODS[b.name] = tsa.build(b.name, b.ss)
    res = oracle_target(b, par, w0)
    assert res.status == 0
    dW, clear = tsa.active_set_jacobian(TargetNlp(b.ss, b.oracle), _SMODS[b.name], res, par, gap=gap)
    return dW, clear, res


def cases(b, count=6, seed=0):
    rng = np.random.default_rng(seed)
    pars = np.array([target_par(b)] + [target_par(b, rng) for _ in range(count - 1)])
    return pars, np.array([target_guess(b, par) for par in pars])


# ---- (1) the anchor agrees with finite differences of the oracle -----------------------------------------------------
def test_target_anchor_matches_oracle_finite_differences(nmpc):
    import target_sens_anchor as tsa
    idx = tsa.theta_ss_index(nmpc.ss)
    pars, w0s = cases(nmpc, 4)
    checked = 0
    for par, w0 in zip(pars, w0s):
        dW, clear, res = anchor(nmpc, par, w0)
        if not clear:
            continue
        fd = np.zeros_like(dW)
        for t, pi in enumerate(idx):
            h = 1e-5 * max(1.0, abs(par[pi]))
            pp, pm = par.copy(), par.copy()
            pp[pi] += h; pm[pi] -= h
            fd[:, t] = (oracle_target(nmpc, pp, res.x).x - oracle_target(nmpc, pm, res.x).x) / (2 * h)
        assert np.abs(fd).max() > 1e-2
        assert np.all(_col_close(dW, fd, 1e-6)), np.abs(fd - dW).max(axis=0)
        checked += 1
    assert checked >= 2


# ---- (2) the device arithmetic matches the anchor -------------------------------------------------------------------
PROBLEMS = ["nmpc_cstr", "nmpc_cstr_ss_user", "nmpc_dis", "lmpc_wb", "enmpc_reactor"]


@pytest.mark.parametrize("name", PROBLEMS)
def test_harness_jacobian_matches_active_set_anchor(name):
    b = _bundle(name)
    p = b.prob
    nth = n_theta_ss(p)
    assert b.lib["gen"]["defines"]["MPCB_SENS_TGT"] == 1
    pars, w0s = cases(b)
    r = harness_tgt(b, pars, w0s, unit_dirs(len(pars), nth))
    checked = 0
    for i, par in enumerate(pars):
        if r["status"][i] != 0:
            continue
        dW, clear, _ = anchor(b, par, r["w"][i], gap=1e-3)
        if not clear:
            continue
        assert r["sstatus"][i] == 0
        J = r["dw"][i].T                                       # [nwss, ntheta_ss]
        assert np.all(_col_close(J, dW, 1e-6)), (name, np.abs(J - dW).max(axis=0))
        checked += 1
    assert checked >= 1, name
    dw = r["dw"][r["sstatus"] == 0]
    assert np.abs(dw).max() > 1e-3
    o = p.nu + p.ny + p.nx + p.nd                              # the Us_prev columns (Delta-u cost, or lam) are not trivial
    assert np.abs(dw[:, o:o + p.nu]).max() > 1e-4


# ---- (3) an anchor that shares nothing with the oracle: lmpc_cstr's target problem is an equality-constrained QP -----
def test_lmpc_cstr_target_jacobian_is_the_qp_kkt_solution(lmpc_cstr):
    """With inactive bounds lmpc_cstr's target problem is min 1/2 |ys - ysp|_Qss^2 + 1/2 |us - usp|_Rss^2 subject to
    xs = A xs + B us + Bd d + px and ys = C xs + Cd d + py + lam (us - Us_prev): its KKT system gives dwss/dtheta_ss
    exactly."""
    b = lmpc_cstr
    p, ns = b.prob, b.prob.ns
    n, m, q, nd = p.nx, p.nu, p.ny, p.nd
    A, Bm, C, Bd, Cd, Qss, Rss = [np.asarray(ns[k], dtype=float) for k in ("A", "B", "C", "Bd", "Cd", "Qss", "Rss")]
    assert p.npx == n and p.npy == q
    rng = np.random.default_rng(5)
    lam = 0.1 * rng.uniform(-1, 1, (q, m))
    pars = []
    for _ in range(3):
        par = target_par(b, rng)
        par[b.ss.off["lam"]:b.ss.off["lam"] + q * m] = lam.reshape(-1, order="F")
        pars.append(par)
    pars = np.array(pars)
    nv, nth = n + m + q, n_theta_ss(p)
    H = np.zeros((nv, nv)); H[n:n + m, n:n + m] = Rss; H[n + m:, n + m:] = Qss
    E = np.zeros((n + q, nv))
    E[:n, :n] = A - np.eye(n); E[:n, n:n + m] = Bm
    E[n:, :n] = C; E[n:, n:n + m] = lam; E[n:, n + m:] = -np.eye(q)
    # theta_ss = [usp | ysp | xsp | d | Us_prev | px | py]: the gradient -[0; Rss usp; Qss ysp] and the right-hand
    # sides of E v
    Ht = np.zeros((nv, nth)); Et = np.zeros((n + q, nth))
    Ht[n:n + m, 0:m] = Rss; Ht[n + m:, m:m + q] = Qss
    o_d, o_u = m + q + n, m + q + n + nd
    o_px = o_u + m
    Et[:n, o_d:o_d + nd] = -Bd; Et[n:, o_d:o_d + nd] = -Cd; Et[n:, o_u:o_u + m] = lam
    Et[:n, o_px:o_px + n] = -np.eye(n); Et[n:, o_px + n:o_px + n + q] = -np.eye(q)
    K = np.block([[H, E.T], [E, np.zeros((n + q, n + q))]])
    T = np.linalg.solve(K, np.vstack([Ht, Et]))[:nv]
    r = harness_tgt(b, pars, np.array([target_guess(b, par) for par in pars]), unit_dirs(len(pars), nth))
    assert np.all(r["status"] == 0) and np.all(r["sstatus"] == 0)
    for i in range(len(pars)):
        assert np.all(_col_close(r["dw"][i].T, T, 1e-8)), np.abs(r["dw"][i].T - T).max(axis=0)
    assert np.abs(T[:, o_u:o_u + m]).max() > 1e-3              # lam (us - Us_prev) makes the Us_prev columns non-trivial


# ---- (4) adjoint consistency -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", PROBLEMS + ["lmpc_cstr"])
def test_target_vjp_is_the_adjoint_of_the_jvp(name):
    b = _bundle(name)
    p = b.prob
    nth = n_theta_ss(p)
    pars, w0s = cases(b)
    rng = np.random.default_rng(11)
    B = len(pars)
    dth = rng.standard_normal((B, 1, nth)); gw = rng.standard_normal((B, b.ss.nw))
    r = harness_tgt(b, pars, w0s, dth, gw)
    ok = r["sstatus"] == 0
    assert ok.sum() >= 1
    lhs = np.einsum("bw,bw->b", gw, r["dw"][:, 0]); rhs = np.einsum("bt,bt->b", r["gth"], dth[:, 0])
    assert np.all(np.abs(lhs - rhs)[ok] <= 1e-10 * np.maximum(np.abs(lhs), np.abs(rhs))[ok])


# ---- (5) failure statuses --------------------------------------------------------------------------------------------
def test_infeasible_target_gives_status_1_and_nan(lmpc_cstr):
    """Bounds that pin xs and us to a point that is not a steady state of the model."""
    b = lmpc_cstr
    p, ss = b.prob, b.ss
    par = target_par(b)
    lbx, ubx = ss.w_lb.copy(), ss.w_ub.copy()
    lbx[:p.nx + p.nu] = 1.0; ubx[:p.nx + p.nu] = 1.0 + 1e-6
    r = harness_tgt(b, par, target_guess(b, par), unit_dirs(1, n_theta_ss(p)), np.ones((1, ss.nw)), lbx=lbx, ubx=ubx,
                    tol=1e-8)
    assert r["status"][0] not in (0, 1) and r["sstatus"][0] == 1
    assert np.all(np.isnan(r["dw"])) and np.all(np.isnan(r["gth"]))


def test_dense_models_are_refused_and_contform_is_not():
    """A large model on the dense derivative path has no target sensitivities (its entry points return < 0, checked
    without a device); enmpc_reactor, whose OCP refuses p, has them."""
    from mpc_code_b200.devicegen import DENSE_SH_ENTRIES, generate_header
    from mpc_code_b200.problem import build_problem, make_specs
    from mpc_code_b200.synthetic import synthetic_namespace
    prob = build_problem(synthetic_namespace(20, 6, 20))
    assert prob.Fx_model.meta.get("kind") == "rk4" and prob.nx * (prob.nx + prob.nu) > DENSE_SH_ENTRIES
    ss, ocp = make_specs(prob)
    assert generate_header(prob, ss, ocp)["defines"]["MPCB_SENS_TGT"] == 0
    enmpc = _bundle("enmpc_reactor").lib["gen"]["defines"]
    assert enmpc["MPCB_SENS_P"] == 0 and enmpc["MPCB_SENS_TGT"] == 1
    lib = ctypes.CDLL(_bundle("nmpc_cstr").lib["so"])
    lib.mpcb_target_sens_size.restype = ctypes.c_long
    assert lib.mpcb_target_sens_size() > 0


# ---- (6) composed gains: target, then OCP ----------------------------------------------------------------------------
def test_composed_gains_match_finite_differences_of_the_oracle_chain(nmpc):
    """dU_0/dd_hat and dU_0/dysp of nmpc_cstr through x_s, u_s: the harness target Jacobian composed in NumPy with the
    OCP's theta and p harnesses, against central differences of the oracle's target solve followed by its OCP solve."""
    p, ss, ocp = nmpc.prob, nmpc.ss, nmpc.ocp
    n, m, nd, q = p.nx, p.nu, p.nd, p.ny
    base = G["ocp_par"][0].copy()
    w0 = G["ocp_w0"]
    par_ss = target_par(nmpc)
    par_ss[ss.off["d"]:ss.off["d"] + nd] = base[ocp.off["d"]:ocp.off["d"] + nd]
    wg = target_guess(nmpc, par_ss)

    def chain(ps):
        ws = oracle_target(nmpc, ps, wg)
        assert ws.status == 0
        par = base.copy()
        par[ocp.off["xs"]:ocp.off["xs"] + n] = ws.x[:n]
        par[ocp.off["us"]:ocp.off["us"] + m] = ws.x[n:n + m]
        par[ocp.off["d"]:ocp.off["d"] + nd] = ps[ss.off["d"]:ss.off["d"] + nd]
        res, _, _ = oracle_solve(nmpc, par, w0)
        assert res.status == 0
        return ws.x, par, res.x[n:n + m]

    wss, par, _ = chain(par_ss)
    nth, nthss = 2 * (n + m), n_theta_ss(p)
    rt = harness_tgt(nmpc, par_ss, wg, unit_dirs(1, nthss))
    assert rt["sstatus"][0] == 0 and np.abs(rt["w"][0] - wss).max() < 1e-8
    T = rt["dw"][0].T[:n + m]                                   # d[xs; us]/dtheta_ss
    ro = harness_sens(nmpc, par, w0, unit_dirs(1, nth))
    Jth = ro["dw"][0].T[n:n + m, n:2 * n + m]                   # dU_0/d[xs; us]
    npp = nd + (p.npx + p.npy) * p.N
    rp = harness_sens_p(nmpc, par, w0, unit_dirs(1, npp))
    Jp = rp["dw"][0].T[n:n + m, :nd]                            # dU_0/dd at fixed targets
    assert ro["sstatus"][0] == 0 and rp["sstatus"][0] == 0
    o_d, o_y = m + q + n, m
    gain_d = Jp + Jth @ T[:, o_d:o_d + nd]
    gain_y = Jth @ T[:, o_y:o_y + q]
    for gain, off, cnt in ((gain_d, ss.off["d"], nd), (gain_y, ss.off["ysp"], q)):
        fd = np.zeros((m, cnt))
        for j in range(cnt):
            h = 1e-5 * max(1.0, abs(par_ss[off + j]))
            pp, pm = par_ss.copy(), par_ss.copy()
            pp[off + j] += h; pm[off + j] -= h
            fd[:, j] = (chain(pp)[2] - chain(pm)[2]) / (2 * h)
        assert np.abs(fd).max() > 1e-3
        assert np.all(_col_close(gain, fd, 1e-5)), np.abs(gain - fd).max(axis=0)
    assert np.abs(Jth @ T[:, o_d:o_d + nd]).max() > 1e-2 * np.abs(Jp).max()   # the target part is not negligible


# ==== on the device ===================================================================================================
def _device_target(b, batch, **opts):
    from mpc_code_b200.solvers import BatchedNlpSolver, MpcbHandle, MpcbLibrary
    h = MpcbHandle(MpcbLibrary(b.lib["so"]), batch, opts_ss=opts or None)
    return h, BatchedNlpSolver("target", b.ss).attach(h)


def _ss_batch(b, B, seed=0):
    """B target problems of Ex_NMPC: the golden instances with perturbed output set-points and disturbance estimates."""
    off, p = b.ss.off, b.prob
    rng = np.random.default_rng(seed)
    par = G["ss_par"][np.arange(B) % G["ss_par"].shape[0]].copy()
    par[:, off["ysp"]:off["ysp"] + p.ny] *= 1 + 0.01 * rng.uniform(-1, 1, (B, p.ny))
    par[:, off["d"]:off["d"] + p.nd] *= 1 + 0.01 * rng.uniform(-1, 1, (B, p.nd))
    return par, G["ss_w0"][np.arange(B) % G["ss_w0"].shape[0]].copy()


@pytest.mark.gpu
def test_device_matches_harness_on_ex_nmpc(nmpc):
    import torch
    B, nth, nw = 4096, n_theta_ss(nmpc.prob), nmpc.ss.nw
    par, w0 = _ss_batch(nmpc, B)
    h, solver = _device_target(nmpc, B)
    sol = solver(x0=w0, p=par)
    sens = solver.sensitivity()
    J = sens.jacobian().cpu().numpy()                                   # [B, nw, nth]
    gw = np.random.default_rng(2).standard_normal((B, nw))
    gth = sens.vjp(gw).cpu().numpy()
    st, sst = solver.stats()["status"].cpu().numpy(), sens.status.cpu().numpy()
    o = h.opts_ss
    idx = np.arange(0, B, B // 64)
    r = harness_tgt(nmpc, par[idx], w0[idx], unit_dirs(len(idx), nth), gw[idx], tol=o.tol, max_iter=o.max_iter,
                    mu_init=o.mu_init, relax=o.bound_relax_factor, honor=o.honor_original_bounds)
    assert np.array_equal(r["status"], st[idx]) and np.array_equal(r["sstatus"], sst[idx])
    ok = r["sstatus"] == 0
    assert ok.sum() >= 32
    assert np.abs(sol["x"].cpu().numpy()[idx] - r["w"]).max() < 1e-9
    for j in np.where(ok)[0]:
        assert np.all(_col_close(J[idx[j]], r["dw"][j].T, 1e-9)), np.abs(J[idx[j]] - r["dw"][j].T).max()
        assert np.allclose(gth[idx[j]], r["gth"][j], rtol=1e-9, atol=1e-9 * np.abs(r["gth"][j]).max())
    assert np.all(np.isnan(J[sst != 0])) and np.all(~np.isnan(J[sst == 0]))
    assert torch.equal(sens.jvp(torch.eye(nth, dtype=torch.float64, device=h.device)[None, 3].expand(B, -1)),
                       sens.jacobian()[:, :, 3])


@pytest.mark.gpu
def test_device_jvp_matches_device_finite_differences(nmpc):
    import target_sens_anchor as tsa
    pars, w0 = _ss_batch(nmpc, 4, seed=3)
    idx = tsa.theta_ss_index(nmpc.ss)
    nb, nth = len(pars), len(idx)
    steps = 1e-5 * np.maximum(1.0, np.abs(pars[:, idx]))
    rows = [pars]
    for sgn in (1, -1):
        for t, pi in enumerate(idx):
            q = pars.copy(); q[:, pi] += sgn * steps[:, t]; rows.append(q)
    allp = np.concatenate(rows)
    allw = np.concatenate([w0] * (1 + 2 * nth))
    h, solver = _device_target(nmpc, allp.shape[0], tol=TIGHT, max_iter=200)
    w = solver(x0=allw, p=allp)["x"].cpu().numpy()
    st = solver.stats()["status"].cpu().numpy()
    sens = solver.sensitivity()
    J = sens.jacobian().cpu().numpy()
    sst = sens.status.cpu().numpy()
    checked = 0
    for i in range(nb):
        if not (np.all(st[i::nb] == 0) and sst[i] == 0):
            continue
        fd = np.stack([(w[nb * (1 + t) + i] - w[nb * (1 + nth + t) + i]) / (2 * steps[i, t]) for t in range(nth)], axis=1)
        assert np.all(_col_close(J[i], fd, 1e-5)), np.abs(J[i] - fd).max(axis=0)
        checked += 1
    assert checked >= 2


@pytest.mark.gpu
def test_capture_repeats_the_solve_bit_for_bit(nmpc):
    import torch
    B = 256
    par, w0 = _ss_batch(nmpc, B, seed=1)
    h, solver = _device_target(nmpc, B)
    w0_t = h.tensor(w0, nmpc.ss.nw)
    keep = w0_t.clone()
    out1 = solver(x0=w0_t, p=par)
    x1, f1 = out1["x"].clone(), out1["f"].clone()
    st1, it1 = solver.stats()["status"].clone(), solver.stats()["iter_count"].clone()
    sens = solver.sensitivity()
    assert torch.equal(sens.wss, x1)                                   # the capture's solution is mpcb_target's output
    assert torch.equal(sens.fac[:, 1].to(torch.int32), st1)
    assert torch.equal(w0_t, keep)                                     # the guess is not modified
    out2 = solver(x0=w0_t, p=par)                                      # and the target solve is unchanged after it
    assert torch.equal(out2["x"], x1) and torch.equal(out2["f"], f1)
    assert torch.equal(solver.stats()["status"], st1) and torch.equal(solver.stats()["iter_count"], it1)
    with pytest.raises(ValueError):
        solver.sensitivity(params=True)


@pytest.mark.gpu
def test_target_layer_gradient_matches_finite_differences(nmpc):
    import torch
    from mpc_code_b200.sensitivity import TargetLayer, theta_ss_of
    p = nmpc.prob
    par, w0 = _ss_batch(nmpc, 4, seed=4)
    pars = torch.as_tensor(par, device="cuda")
    w0 = torch.as_tensor(w0, device="cuda")
    h, solver = _device_target(nmpc, 4, tol=TIGHT, max_iter=200)
    layer = TargetLayer(solver)
    theta = theta_ss_of(pars, p.nx, p.nu, p.ny, p.nd).clone().requires_grad_(True)

    def loss_of(th):
        w = layer(th, pars, w0)
        return (w[:, :p.nx + p.nu] ** 2).sum(dim=1)                     # |x_s|^2 + |u_s|^2, per instance

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
def test_controller_gains(nmpc):
    """x_hat is the feedback gain; d_hat is the total derivative of U_0 through the target problem and the OCP, checked
    against central differences of a target + OCP re-solve at d_hat +- h (status-0 instances)."""
    import torch
    from mpc_code_b200.mpc_loop import INFEASIBLE, CompiledProblem
    p = nmpc.prob
    n, m, nd = p.nx, p.nu, p.nd
    cp = CompiledProblem(p, "nmpc_cstr")
    B = 16
    tight = dict(tol=TIGHT, max_iter=200)
    ctl = cp.controller(B, opts_ss=tight, opts_dyn=tight)
    ctl.step()
    ctl.step()
    gains = ctl.controller_gains()
    assert torch.equal(gains["x_hat"], ctl.feedback_gain()) and gains["u_prev"] is None
    assert gains["d_hat"].shape == (B, m, nd) and gains["ysp"].shape == (B, m, p.ny)
    par_ss, wss0 = ctl.solver_ss._last_target
    par_ocp, _ = ctl.solver._last_ocp
    w_guess = ctl.w_guess.clone()
    st_ss = ctl.solver_ss.stats()["status"].clone()
    st_ocp = ctl.solver.stats()["status"].clone()
    off, offs = cp.ocp_spec.off, cp.ss_spec.off
    h = ctl.h

    def u0_at(ps):
        wss, _, sts, _ = h.target(ps, wss0)
        par = par_ocp.clone()
        use = (sts != INFEASIBLE).unsqueeze(1)
        par[:, off["xs"]:off["xs"] + n] = torch.where(use, wss[:, :n], par[:, off["xs"]:off["xs"] + n])
        par[:, off["us"]:off["us"] + m] = torch.where(use, wss[:, n:n + m], par[:, off["us"]:off["us"] + m])
        par[:, off["d"]:off["d"] + nd] = ps[:, offs["d"]:offs["d"] + nd]
        w, _, st, _ = h.ocp(par, w_guess)
        return w[:, n:n + m], (sts == 0) & (st == 0)

    fd = torch.zeros(B, m, nd, dtype=torch.float64, device=h.device)
    ok = (st_ss == 0) & (st_ocp == 0)
    for j in range(nd):
        step = 1e-5 * torch.clamp(par_ss[:, offs["d"] + j].abs(), min=1.0)
        pp, pm = par_ss.clone(), par_ss.clone()
        pp[:, offs["d"] + j] += step; pm[:, offs["d"] + j] -= step
        (up, okp), (um, okm) = u0_at(pp), u0_at(pm)
        fd[:, :, j] = (up - um) / (2 * step.unsqueeze(1))
        ok &= okp & okm
    assert int(ok.sum()) >= B // 2
    G_, F_ = gains["d_hat"][ok].cpu().numpy(), fd[ok].cpu().numpy()
    for i in range(G_.shape[0]):
        assert np.all(_col_close(G_[i], F_[i], 1e-5)), (G_[i], F_[i])
    ctl2 = cp.controller(4)
    ctl2.step_fused()
    with pytest.raises(RuntimeError, match="step_fused"):
        ctl2.controller_gains()
    with pytest.raises(NotImplementedError, match="fused step"):
        ctl2.solver_ss.sensitivity()
